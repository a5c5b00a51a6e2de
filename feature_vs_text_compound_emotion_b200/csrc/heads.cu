// fp32 building blocks for the alternative fusion heads of the reference (CAN, JMT, MT;
// models/model.py:529-684, :709-750, :895-1167): nn.Linear, the AttentionFusion gate, single-head
// scaled-dot-product attention over a sequence (nn.MultiheadAttention(E, 1)), residual + LayerNorm.
// C-ABI: cer_linear_forward, cer_softmax_gate, cer_sdpa_forward (exact fp32, CUDA cores), cer_sdpa_tc_forward
// (TF32 tensor-core flash attention, the default of the mirrors), cer_add_layernorm.
// These heads are ~0.1 % of the path's FLOPs and latency bound; the linear layers share the packed-FFMA2
// row GEMM of the training plan.
#include <cuda_runtime.h>
#include <cstdint>

#include "../../include/cer_b200.h"
#include "common.h"
#include "row_gemm.h"

namespace cer {

// out[r, :] = softmax(gate[r, :]) * feat[r, :]    (AttentionFusion.forward, model.py:563-567)
__global__ void __launch_bounds__(256) softmax_gate_kernel(const float* __restrict__ gate, const float* __restrict__ feat,
                                                           int rows, int dim, float* __restrict__ out) {
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float* g = gate + (long long)r * dim;
  float mx = -3.4e38f;
  for (int i = lane; i < dim; i += 32) mx = fmaxf(mx, g[i]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float s = 0.f;
  for (int i = lane; i < dim; i += 32) s += expf(g[i] - mx);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float inv = 1.f / s;
  for (int i = lane; i < dim; i += 32) out[(long long)r * dim + i] = expf(g[i] - mx) * inv * feat[(long long)r * dim + i];
}

// Single-head attention: out[b, i, :] = softmax_j(q[b,i,:] . k[b,j,:] / sqrt(E)) v[b,j,:].
// One warp per query row: lanes stride over the keys for the scores (kept in shared memory), then
// over the E output features.  E <= 128 * 4, len_k <= 4096 (scores in smem).
__global__ void __launch_bounds__(256) sdpa_kernel(const float* __restrict__ q, int ldq, const float* __restrict__ k, int ldk,
                                                   const float* __restrict__ v, int ldv, int len_q, int len_k, int E,
                                                   float* __restrict__ out, int ldo) {
  extern __shared__ float sm_f[];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* s_q = sm_f + w * (E + ((len_k + 3) & ~3));       // [E], 16-byte aligned per warp
  float* s_p = s_q + E;                      // [len_k]
  const int b = blockIdx.y;
  const int i = blockIdx.x * 8 + w;
  if (i >= len_q) return;
  const float* qp = q + ((long long)b * len_q + i) * ldq;
  for (int d = lane; d < E; d += 32) s_q[d] = qp[d];
  __syncwarp();
  const float scale = rsqrtf((float)E);
  const float* kb = k + (long long)b * len_k * ldk;
  float mx = -3.4e38f;
  for (int j = lane; j < len_k; j += 32) {
    const float4* kp = reinterpret_cast<const float4*>(kb + (long long)j * ldk);
    float s = 0.f;
    for (int d = 0; d < E / 4; ++d) {
      const float4 kk = __ldg(kp + d);
      const float4 qq = *reinterpret_cast<const float4*>(s_q + 4 * d);
      s = fmaf(qq.x, kk.x, s); s = fmaf(qq.y, kk.y, s); s = fmaf(qq.z, kk.z, s); s = fmaf(qq.w, kk.w, s);
    }
    s *= scale;
    s_p[j] = s;
    mx = fmaxf(mx, s);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float den = 0.f;
  for (int j = lane; j < len_k; j += 32) { const float e = expf(s_p[j] - mx); s_p[j] = e; den += e; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) den += __shfl_xor_sync(0xffffffffu, den, o);
  __syncwarp();
  const float inv = 1.f / den;
  const float* vb = v + (long long)b * len_k * ldv;
  float* op = out + ((long long)b * len_q + i) * ldo;
  for (int d = lane; d < E; d += 32) {
    float acc = 0.f;
    for (int j = 0; j < len_k; ++j) acc = fmaf(s_p[j], __ldg(vb + (long long)j * ldv + d), acc);
    op[d] = acc * inv;
  }
}

// ------------------------------------------------------------------------------------------
// The same attention on the tensor cores: flash-attention forward with warp-level TF32 MMAs
// (mma.sync.m16n8k8, fp32 accumulate) and an online softmax in fp32 registers.  The head's attention is
// 0.1 % of the path and latency bound (nn.MultiheadAttention(128, 1) over T = 300, and over all L*B
// positions in the final encoder, models/model.py:731, :917-931, :1003-1012), so the warp-level MMA -- no
// TMEM, no descriptors -- is the right tool; it still removes the 2 * L * E FMAs per query of sdpa_kernel.
//   CTA = 4 warps x 16 queries; keys in blocks of 64; Q / K / V tiles in shared memory as tf32
//   (cvt.rna), row stride E + 4 floats so every fragment load is bank-conflict free.
//   P (the S accumulators) feeds the second MMA without a shuffle: inside each 8-key tile the k index
//   of the P.V product is permuted (A column t <-> key 2t, column t+4 <-> key 2t+1), and the V fragment
//   uses the same permutation -- a sum over keys does not care about their order.
// ------------------------------------------------------------------------------------------
constexpr int kSdpaQ = 64, kSdpaK = 64;

__device__ __forceinline__ uint32_t f2tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ void mma_tf32(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

//   kSeg: blockIdx.y is a segment s; q, k, v and out rows are [seg_off[s], seg_off[s+1]) of their buffers and
//   len_q = len_k = that length (self- or cross-attention inside one video of a concatenated batch).  A CTA past
//   its segment's end returns before any load or barrier; every other instruction is the uniform kernel's, so a
//   segment gives the same bits as a batch-1 launch on it alone.
//   kHeads (segmented only): blockIdx.z is a head h; q, k, v and out start E * h columns further into their rows
//   (head h of a multi-head projection through the same row pitches).  Otherwise the code is kSeg's.
template <int E, bool kSeg, bool kHeads = false>
__global__ void __launch_bounds__(128) sdpa_tc_kernel(const float* __restrict__ q, int ldq, const float* __restrict__ k, int ldk,
                                                      const float* __restrict__ v, int ldv, int len_q, int len_k,
                                                      float* __restrict__ out, int ldo, const int* __restrict__ seg_off) {
  constexpr int LD = E + 4;
  extern __shared__ float sm_f[];
  uint32_t* sQ = reinterpret_cast<uint32_t*>(sm_f);            // [64][LD] tf32 bits
  uint32_t* sK = sQ + kSdpaQ * LD;
  uint32_t* sV = sK + kSdpaK * LD;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int b = blockIdx.y;
  const int q0 = blockIdx.x * kSdpaQ;
  long long row_q, row_k;
  if constexpr (kSeg) {
    row_q = row_k = seg_off[b];
    len_q = len_k = seg_off[b + 1] - seg_off[b];
    if (q0 >= len_q) return;                                    // uniform per CTA: no barrier is reached by part of it
  } else {
    row_q = (long long)b * len_q;
    row_k = (long long)b * len_k;
  }
  if constexpr (kHeads) {
    static_assert(kSeg, "head batching is a form of the segmented kernel");
    const int col = E * blockIdx.z;
    q += col; k += col; v += col; out += col;
  }
  const float* qb = q + row_q * ldq;
  const float* kb = k + row_k * ldk;
  const float* vb = v + row_k * ldv;
  const float scale = rsqrtf((float)E);

  for (int i = threadIdx.x; i < kSdpaQ * (E / 4); i += 128) {
    const int r = i / (E / 4), c = (i - r * (E / 4)) * 4;
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    if (q0 + r < len_q) x = *reinterpret_cast<const float4*>(qb + (long long)(q0 + r) * ldq + c);
    uint32_t* d = sQ + r * LD + c;
    d[0] = f2tf32(x.x * scale); d[1] = f2tf32(x.y * scale); d[2] = f2tf32(x.z * scale); d[3] = f2tf32(x.w * scale);
  }
  float o[E / 8][4];
#pragma unroll
  for (int n = 0; n < E / 8; ++n) { o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f; }
  float mrow[2] = {-3.0e38f, -3.0e38f}, lrow[2] = {0.f, 0.f};   // rows g and g + 8 of this warp's 16 queries
  const uint32_t* wq = sQ + (warp * 16) * LD;

  for (int k0 = 0; k0 < len_k; k0 += kSdpaK) {
    __syncthreads();                                            // previous block's K / V fully consumed (and Q written)
    for (int i = threadIdx.x; i < kSdpaK * (E / 4); i += 128) {
      const int r = i / (E / 4), c = (i - r * (E / 4)) * 4;
      float4 x = make_float4(0.f, 0.f, 0.f, 0.f), y = x;
      if (k0 + r < len_k) {
        x = __ldg(reinterpret_cast<const float4*>(kb + (long long)(k0 + r) * ldk + c));
        y = __ldg(reinterpret_cast<const float4*>(vb + (long long)(k0 + r) * ldv + c));
      }
      uint32_t* dk = sK + r * LD + c;
      uint32_t* dv = sV + r * LD + c;
      dk[0] = f2tf32(x.x); dk[1] = f2tf32(x.y); dk[2] = f2tf32(x.z); dk[3] = f2tf32(x.w);
      dv[0] = f2tf32(y.x); dv[1] = f2tf32(y.y); dv[2] = f2tf32(y.z); dv[3] = f2tf32(y.w);
    }
    __syncthreads();
    // S = (Q * scale) K^T : 16 x 64 per warp
    float sc[kSdpaK / 8][4];
#pragma unroll
    for (int n = 0; n < kSdpaK / 8; ++n) { sc[n][0] = sc[n][1] = sc[n][2] = sc[n][3] = 0.f; }
#pragma unroll
    for (int kk = 0; kk < E / 8; ++kk) {
      const uint32_t a0 = wq[g * LD + kk * 8 + t], a1 = wq[(g + 8) * LD + kk * 8 + t];
      const uint32_t a2 = wq[g * LD + kk * 8 + t + 4], a3 = wq[(g + 8) * LD + kk * 8 + t + 4];
#pragma unroll
      for (int n = 0; n < kSdpaK / 8; ++n) {
        const uint32_t* kr = sK + (n * 8 + g) * LD + kk * 8 + t;
        mma_tf32(sc[n], a0, a1, a2, a3, kr[0], kr[4]);
      }
    }
    // online softmax (fp32): this thread holds columns 2t, 2t+1 of every 8-key tile for rows g and g+8
    float mx[2] = {mrow[0], mrow[1]};
#pragma unroll
    for (int n = 0; n < kSdpaK / 8; ++n) {
      const int key = k0 + n * 8 + 2 * t;
      if (key >= len_k) { sc[n][0] = -3.0e38f; sc[n][2] = -3.0e38f; }
      if (key + 1 >= len_k) { sc[n][1] = -3.0e38f; sc[n][3] = -3.0e38f; }
      mx[0] = fmaxf(mx[0], fmaxf(sc[n][0], sc[n][1]));
      mx[1] = fmaxf(mx[1], fmaxf(sc[n][2], sc[n][3]));
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
    }
    const float corr0 = __expf(mrow[0] - mx[0]), corr1 = __expf(mrow[1] - mx[1]);
    mrow[0] = mx[0]; mrow[1] = mx[1];
    float sum0 = 0.f, sum1 = 0.f;
    uint32_t pa[kSdpaK / 8][4];                                 // P as A fragments (k permuted inside each tile)
#pragma unroll
    for (int n = 0; n < kSdpaK / 8; ++n) {
      const float p0 = __expf(sc[n][0] - mx[0]), p1 = __expf(sc[n][1] - mx[0]);
      const float p2 = __expf(sc[n][2] - mx[1]), p3 = __expf(sc[n][3] - mx[1]);
      sum0 += p0 + p1; sum1 += p2 + p3;
      pa[n][0] = f2tf32(p0);      // row g,   A column t     <-> key 2t
      pa[n][1] = f2tf32(p2);      // row g+8, A column t
      pa[n][2] = f2tf32(p1);      // row g,   A column t + 4 <-> key 2t + 1
      pa[n][3] = f2tf32(p3);      // row g+8, A column t + 4
    }
    lrow[0] = lrow[0] * corr0 + sum0;
    lrow[1] = lrow[1] * corr1 + sum1;
#pragma unroll
    for (int n = 0; n < E / 8; ++n) { o[n][0] *= corr0; o[n][1] *= corr0; o[n][2] *= corr1; o[n][3] *= corr1; }
    // O += P V : k runs over the 64 keys of the block (8 tiles), n over the E features
#pragma unroll
    for (int kt = 0; kt < kSdpaK / 8; ++kt) {
      const uint32_t* vr = sV + (kt * 8 + 2 * t) * LD + g;
#pragma unroll
      for (int n = 0; n < E / 8; ++n) mma_tf32(o[n], pa[kt][0], pa[kt][1], pa[kt][2], pa[kt][3], vr[n * 8], vr[LD + n * 8]);
    }
  }
  // row sums live in 4 lanes each
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    lrow[r] += __shfl_xor_sync(0xffffffffu, lrow[r], 1);
    lrow[r] += __shfl_xor_sync(0xffffffffu, lrow[r], 2);
  }
  const float inv0 = 1.f / lrow[0], inv1 = 1.f / lrow[1];
  const int r0 = q0 + warp * 16 + g, r1 = r0 + 8;
  float* ob = out + row_q * ldo;
#pragma unroll
  for (int n = 0; n < E / 8; ++n) {
    if (r0 < len_q) *reinterpret_cast<float2*>(ob + (long long)r0 * ldo + n * 8 + 2 * t) = make_float2(o[n][0] * inv0, o[n][1] * inv0);
    if (r1 < len_q) *reinterpret_cast<float2*>(ob + (long long)r1 * ldo + n * 8 + 2 * t) = make_float2(o[n][2] * inv1, o[n][3] * inv1);
  }
}

// out[r, :] = LayerNorm(x[r, :] + res[r, :]) * gamma + beta   (res may be null), one warp per row
__global__ void __launch_bounds__(256) add_layernorm_kernel(const float* __restrict__ x, const float* __restrict__ res,
                                                            int rows, int dim, const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, float eps,
                                                            float* __restrict__ out) {
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float* xp = x + (long long)r * dim;
  const float* rp = res ? res + (long long)r * dim : nullptr;
  float s = 0.f;
  for (int i = lane; i < dim; i += 32) s += xp[i] + (rp ? rp[i] : 0.f);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s / dim;
  float ss = 0.f;
  for (int i = lane; i < dim; i += 32) { const float d = xp[i] + (rp ? rp[i] : 0.f) - mean; ss += d * d; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const float rstd = 1.f / sqrtf(ss / dim + eps);
  for (int i = lane; i < dim; i += 32)
    out[(long long)r * dim + i] = (xp[i] + (rp ? rp[i] : 0.f) - mean) * rstd * gamma[i] + beta[i];
}

// a += b (gradient accumulation where two branches meet)
__global__ void add_inplace_kernel(float* __restrict__ a, const float* __restrict__ b, long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) a[i] += b[i];
}

// y = tanh(y) in place (the REGRESSION task's output squashing, models/model.py:523, :682, :1165)
__global__ void tanh_inplace_kernel(float* __restrict__ y, long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    y[i] = tanhf(y[i]);
}

}  // namespace cer

using namespace cer;

extern "C" int cer_linear_forward(const float* x_dev, int64_t rows, int32_t in_dim, int32_t ldx, const float* w_dev,
                                  const float* bias_dev, int32_t out_dim, int32_t act, float* y_dev, int32_t ldy, void* stream) {
  if (!x_dev || !w_dev || !y_dev || rows < 0 || in_dim <= 0 || out_dim <= 0 || ldx < in_dim || ldy < out_dim || act < 0 || act > 2 ||
      rows > (1 << 24))
    return set_error(CER_ERR_INVALID, "cer_linear_forward: bad argument");
  if (rows == 0) return CER_OK;
  int rc = cer_check_device();
  if (rc) return rc;
  RowGemm g{};
  g.A = x_dev; g.lda = ldx; g.B = w_dev; g.C = y_dev; g.ldc = ldy;
  g.R = (int)rows; g.T = (int)rows; g.N = out_dim; g.K = in_dim; g.taps = 1;
  g.bias = bias_dev;
  g.epi = act == 0 ? EPI_LINEAR : (act == 1 ? EPI_LRELU_DROP : EPI_RELU);     // LeakyReLU = LRELU_DROP with p = 0
  g.drop.key = 0; g.drop.thr = 0; g.drop.scale = 1.f;
  return launch_row_gemm(g, false, static_cast<cudaStream_t>(stream));
}

extern "C" int cer_softmax_gate(const float* gate_dev, const float* feat_dev, int64_t rows, int32_t dim, float* out_dev,
                                void* stream) {
  if (!gate_dev || !feat_dev || !out_dev || rows < 0 || dim <= 0 || rows > (1 << 30))
    return set_error(CER_ERR_INVALID, "cer_softmax_gate: bad argument");
  if (rows == 0) return CER_OK;
  softmax_gate_kernel<<<(int)((rows + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(gate_dev, feat_dev, (int)rows, dim,
                                                                                           out_dev);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

extern "C" int cer_sdpa_forward(const float* q_dev, int32_t ldq, const float* k_dev, int32_t ldk, const float* v_dev,
                                int32_t ldv, int32_t batch, int32_t len_q, int32_t len_k, int32_t dim, float* out_dev,
                                int32_t ldo, void* stream) {
  if (!q_dev || !k_dev || !v_dev || !out_dev || batch <= 0 || len_q <= 0 || len_k <= 0 || dim <= 0 || dim % 4 || ldq < dim ||
      ldk < dim || ldv < dim || ldo < dim || ldk % 4 || batch > 65535)
    return set_error(CER_ERR_INVALID, "cer_sdpa_forward: bad argument (dim and ldk must be multiples of 4)");
  if ((reinterpret_cast<uintptr_t>(k_dev) & 15) != 0) return set_error(CER_ERR_INVALID, "cer_sdpa_forward: k must be 16B aligned");
  const size_t smem = (size_t)8 * (dim + ((len_k + 3) & ~3)) * sizeof(float);
  if (smem > 200 * 1024) return set_error(CER_ERR_INVALID, "cer_sdpa_forward: sequence too long for the shared-memory score rows");
  if (smem > 48 * 1024) {
    static unsigned long long configured = 0;
    if (first_use_on_device(&configured))
      CER_CUDA(cudaFuncSetAttribute(sdpa_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  }
  dim3 grid((len_q + 7) / 8, batch);
  sdpa_kernel<<<grid, 256, smem, static_cast<cudaStream_t>(stream)>>>(q_dev, ldq, k_dev, ldk, v_dev, ldv, len_q, len_k, dim,
                                                                     out_dev, ldo);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

// Uniform: grid (ceil(len_q / 64), batch).  Segmented (seg_off != null): grid (ceil(len_q / 64), n_seg, heads), len_q
// the longest segment.
template <int E, bool kSeg, bool kHeads = false>
static int launch_sdpa_tc(const float* q, int ldq, const float* k, int ldk, const float* v, int ldv, int batch, int len_q, int len_k,
                          float* out, int ldo, const int* seg_off, cudaStream_t st, int heads = 1) {
  const size_t smem = (size_t)(kSdpaQ + 2 * kSdpaK) * (E + 4) * sizeof(float);
  static unsigned long long configured = 0;
  if (first_use_on_device(&configured))
    CER_CUDA(cudaFuncSetAttribute(sdpa_tc_kernel<E, kSeg, kHeads>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid((len_q + kSdpaQ - 1) / kSdpaQ, batch, heads);
  sdpa_tc_kernel<E, kSeg, kHeads><<<grid, 128, smem, st>>>(q, ldq, k, ldk, v, ldv, len_q, len_k, out, ldo, seg_off);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

// dim / pitch / alignment conditions shared by both entry points
static int check_sdpa_tc(const char* what, const float* q_dev, int32_t ldq, const float* k_dev, int32_t ldk, const float* v_dev,
                         int32_t ldv, int32_t dim, const float* out_dev, int32_t ldo) {
  if ((dim != 64 && dim != 128) || ldq % 4 || ldk % 4 || ldv % 4 || ldo % 2)
    return set_error(CER_ERR_INVALID, std::string(what) + ": dim must be 64 or 128, row pitches multiples of 4 floats");
  if ((reinterpret_cast<uintptr_t>(q_dev) | reinterpret_cast<uintptr_t>(k_dev) | reinterpret_cast<uintptr_t>(v_dev)) & 15 ||
      reinterpret_cast<uintptr_t>(out_dev) & 7)
    return set_error(CER_ERR_INVALID, std::string(what) + ": q / k / v must be 16-byte aligned, out 8-byte aligned");
  return cer_check_device();
}

extern "C" int cer_sdpa_tc_forward(const float* q_dev, int32_t ldq, const float* k_dev, int32_t ldk, const float* v_dev,
                                   int32_t ldv, int32_t batch, int32_t len_q, int32_t len_k, int32_t dim, float* out_dev,
                                   int32_t ldo, void* stream) {
  if (!q_dev || !k_dev || !v_dev || !out_dev || batch <= 0 || len_q <= 0 || len_k <= 0 || ldq < dim || ldk < dim || ldv < dim ||
      ldo < dim || batch > 65535)
    return set_error(CER_ERR_INVALID, "cer_sdpa_tc_forward: bad argument");
  int rc = check_sdpa_tc("cer_sdpa_tc_forward", q_dev, ldq, k_dev, ldk, v_dev, ldv, dim, out_dev, ldo);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return dim == 128 ? launch_sdpa_tc<128, false>(q_dev, ldq, k_dev, ldk, v_dev, ldv, batch, len_q, len_k, out_dev, ldo, nullptr, st)
                    : launch_sdpa_tc<64, false>(q_dev, ldq, k_dev, ldk, v_dev, ldv, batch, len_q, len_k, out_dev, ldo, nullptr, st);
}

extern "C" int cer_sdpa_tc_seg_forward(const float* q_dev, int32_t ldq, const float* k_dev, int32_t ldk, const float* v_dev,
                                       int32_t ldv, const int32_t* seg_off_dev, int32_t n_seg, int32_t max_len, int32_t dim,
                                       float* out_dev, int32_t ldo, void* stream) {
  if (!q_dev || !k_dev || !v_dev || !out_dev || !seg_off_dev || n_seg < 0 || max_len < 0 || ldq < dim || ldk < dim ||
      ldv < dim || ldo < dim)
    return set_error(CER_ERR_INVALID, "cer_sdpa_tc_seg_forward: bad argument");
  if (n_seg > 65535) return set_error(CER_ERR_INVALID, "cer_sdpa_tc_seg_forward: more than 65535 segments (the grid's y limit)");
  int rc = check_sdpa_tc("cer_sdpa_tc_seg_forward", q_dev, ldq, k_dev, ldk, v_dev, ldv, dim, out_dev, ldo);
  if (rc) return rc;
  if (n_seg == 0 || max_len == 0) return CER_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return dim == 128 ? launch_sdpa_tc<128, true>(q_dev, ldq, k_dev, ldk, v_dev, ldv, n_seg, max_len, max_len, out_dev, ldo, seg_off_dev, st)
                    : launch_sdpa_tc<64, true>(q_dev, ldq, k_dev, ldk, v_dev, ldv, n_seg, max_len, max_len, out_dev, ldo, seg_off_dev, st);
}

extern "C" int cer_sdpa_tc_seg_heads_forward(const float* q_dev, int32_t ldq, const float* k_dev, int32_t ldk, const float* v_dev,
                                             int32_t ldv, const int32_t* seg_off_dev, int32_t n_seg, int32_t max_len, int32_t dim,
                                             int32_t heads, float* out_dev, int32_t ldo, void* stream) {
  if (!q_dev || !k_dev || !v_dev || !out_dev || !seg_off_dev || n_seg < 0 || max_len < 0 || heads <= 0 || heads > 64 ||
      ldq < dim * heads || ldk < dim * heads || ldv < dim * heads || ldo < dim * heads)
    return set_error(CER_ERR_INVALID, "cer_sdpa_tc_seg_heads_forward: bad argument (1 <= heads <= 64, pitches >= dim * heads)");
  if (n_seg > 65535) return set_error(CER_ERR_INVALID, "cer_sdpa_tc_seg_heads_forward: more than 65535 segments (the grid's y limit)");
  if (dim != 64) return set_error(CER_ERR_INVALID, "cer_sdpa_tc_seg_heads_forward: dim must be 64");
  int rc = check_sdpa_tc("cer_sdpa_tc_seg_heads_forward", q_dev, ldq, k_dev, ldk, v_dev, ldv, dim, out_dev, ldo);
  if (rc) return rc;
  if (n_seg == 0 || max_len == 0) return CER_OK;
  return launch_sdpa_tc<64, true, true>(q_dev, ldq, k_dev, ldk, v_dev, ldv, n_seg, max_len, max_len, out_dev, ldo, seg_off_dev,
                                        static_cast<cudaStream_t>(stream), heads);
}

extern "C" int cer_add_layernorm(const float* x_dev, const float* res_dev, int64_t rows, int32_t dim, const float* gamma_dev,
                                 const float* beta_dev, float eps, float* out_dev, void* stream) {
  if (!x_dev || !gamma_dev || !beta_dev || !out_dev || rows < 0 || dim <= 0 || rows > (1 << 30))
    return set_error(CER_ERR_INVALID, "cer_add_layernorm: bad argument");
  if (rows == 0) return CER_OK;
  add_layernorm_kernel<<<(int)((rows + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(x_dev, res_dev, (int)rows, dim,
                                                                                            gamma_dev, beta_dev, eps, out_dev);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

extern "C" int cer_add_inplace(float* a_dev, const float* b_dev, int64_t n, void* stream) {
  if (!a_dev || !b_dev || n < 0) return set_error(CER_ERR_INVALID, "cer_add_inplace: bad argument");
  if (n == 0) return CER_OK;
  const int blocks = (int)((n + 255) / 256 < 148 * 8 ? (n + 255) / 256 : 148 * 8);
  add_inplace_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(a_dev, b_dev, (long long)n);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

extern "C" int cer_tanh_inplace(float* y_dev, int64_t n, void* stream) {
  if (!y_dev || n < 0) return set_error(CER_ERR_INVALID, "cer_tanh_inplace: bad argument");
  if (n == 0) return CER_OK;
  const int blocks = (int)((n + 255) / 256 < 148 * 8 ? (n + 255) / 256 : 148 * 8);
  tanh_inplace_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(y_dev, (long long)n);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}
