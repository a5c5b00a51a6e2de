// CAN fusion head + tail, fused, with every row computed the same way at any row count.
//
// Reference: AttentionFusion.forward (models/model.py:552-568) and the fc1 -> bn1 -> leaky_relu -> fc2 tail of
// CAN.forward (:678-682), per frame:
//   cat = [attn_0(z_0) | ... | attn_{M-1}(z_{M-1})]          (Linear(C_i -> 128) each, D = 128 * M)
//   g   = softmax(weights(cat)) * cat                         (softmax over all D entries)
//   out = fc2(leaky_relu(fc1'(g), 0.01))                      (fc1' = fc1 with the eval bn1 affine folded in)
//   tanh(out) when the task is REGRESSION.
//
// Offline CAN chains cer_linear_forward launches, whose row GEMM picks split-K or a larger tile from the grid size,
// so a row's value depends on how many rows share the call.  A live stream must not change with how many other
// streams share its push, so here every output element is one fp32 accumulator summed over k = 0, 1, ..., K - 1,
// then + bias; the softmax reductions run over fixed index ranges in a fixed order.  Nothing depends on `rows`, on
// the tile a row lands in or on the grid.
//
// A CTA owns a tile of kCanRows frames; its activations stay in shared memory, feature-major ([k][row], so a
// thread reads its 8 rows of one feature with two 16-byte loads).  The weights (~1.4 MB fp32 at the reference's
// sizes: L2-resident, far too large for shared memory) stream through a double-buffered K-chunk with cp.async.
// Thread t owns rows 8 * (t / 64) + 0..7 and columns t % 64 + 64 q: 64 fp32 accumulators, CUDA cores (the result
// must agree with offline CAN's exact fp32 to reordering, which rules out TF32).
#include <cuda_runtime.h>
#include <algorithm>
#include <cmath>
#include <cstdint>

#include "../../include/cer_b200.h"
#include "common.h"

namespace cer {

constexpr int kCanThreads = 256;
constexpr int kCanRows = 32;           // frames per tile = shared-memory row pitch of the activations
constexpr int kCanRowsPerThread = 8;   // kCanThreads / 64 row groups of 8
constexpr int kCanColSteps = 8;        // columns c, c + 64, ..., c + 448: N <= 512
constexpr int kCanKC = 8;              // weight K-chunk
constexpr int kCanMaxDim = 512;        // C_i and D = 128 * M
constexpr int kCanMaxOut = 64;
constexpr int kCanAttn = 128;          // AttentionFusion's num_out_feats in CAN (model.py:601)

struct CanArgs {
  cer_can_head_weights w;
  const float* feat[CER_MAX_MODALS];
  long long ld[CER_MAX_MODALS];
  long long rows;
  int D, c_max, apply_tanh;
};

__device__ __forceinline__ void cp_async4(float* dst, const float* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(dst))),
               "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait1() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }

// Weight columns [k0, k0 + kc) of W [N][K] -> ws [kc][N].  Consecutive threads take consecutive output features
// (conflict-free stores); the 32-byte sectors they leave half-used are the next k's and stay in L1 (.ca).
__device__ __forceinline__ void load_chunk(const float* __restrict__ W, int N, int K, int k0, float* ws) {
  const int kc = min(kCanKC, K - k0);
  for (int i = threadIdx.x; i < N * kc; i += kCanThreads) {
    const int j = i % N, kk = i / N;
    cp_async4(ws + kk * N + j, W + (size_t)j * K + k0 + kk);
  }
}

// act 0: none, 1: LeakyReLU(0.01), 2: tanh.
// Y = act(X W^T + b) over the tile: X feature-major in shared memory [K][kCanRows]; Y either feature-major in shared
// memory (ldy_row = 0) or row-major in global memory (row r at y + r * ldy_row, only rows < valid written).
// Ends with the block synchronised, so Y may be read and X overwritten right after.
__device__ void tile_linear(const float* __restrict__ W, const float* __restrict__ b, int N, int K, const float* xs,
                            float* y, long long ldy_row, long long valid, int act, float* ws) {
  const int rg = threadIdx.x >> 6, c0 = threadIdx.x & 63;
  const int r0 = rg * kCanRowsPerThread;
  const bool live = r0 < valid;            // rows past the end: skip the FMAs, keep the loads and barriers
  float acc[kCanRowsPerThread][kCanColSteps];
#pragma unroll
  for (int i = 0; i < kCanRowsPerThread; ++i)
#pragma unroll
    for (int q = 0; q < kCanColSteps; ++q) acc[i][q] = 0.f;
  const int chunks = (K + kCanKC - 1) / kCanKC;
  const int bufsz = kCanKC * N;
  load_chunk(W, N, K, 0, ws);
  cp_async_commit();
  for (int c = 0; c < chunks; ++c) {
    if (c + 1 < chunks) load_chunk(W, N, K, (c + 1) * kCanKC, ws + ((c + 1) & 1) * bufsz);
    cp_async_commit();                     // possibly empty: wait_group 1 then always means "chunk c has landed"
    cp_async_wait1();
    __syncthreads();
    const float* wc = ws + (c & 1) * bufsz;
    const int k0 = c * kCanKC, kc = min(kCanKC, K - k0);
    if (live) {
      for (int kk = 0; kk < kc; ++kk) {
        const float4 xa = *reinterpret_cast<const float4*>(xs + (size_t)(k0 + kk) * kCanRows + r0);
        const float4 xb = *reinterpret_cast<const float4*>(xs + (size_t)(k0 + kk) * kCanRows + r0 + 4);
        const float xv[kCanRowsPerThread] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
#pragma unroll
        for (int q = 0; q < kCanColSteps; ++q) {
          const int j = c0 + 64 * q;
          if (j < N) {
            const float wv = wc[kk * N + j];
#pragma unroll
            for (int i = 0; i < kCanRowsPerThread; ++i) acc[i][q] = fmaf(xv[i], wv, acc[i][q]);
          }
        }
      }
    }
    __syncthreads();                       // chunk c consumed before chunk c + 2 overwrites its buffer
  }
#pragma unroll
  for (int q = 0; q < kCanColSteps; ++q) {
    const int j = c0 + 64 * q;
    if (j >= N) continue;
    const float bj = __ldg(b + j);
#pragma unroll
    for (int i = 0; i < kCanRowsPerThread; ++i) {
      float v = acc[i][q] + bj;
      if (act == 1) v = v > 0.f ? v : 0.01f * v;
      else if (act == 2) v = tanhf(v);
      if (ldy_row == 0) y[(size_t)j * kCanRows + r0 + i] = v;
      else if (r0 + i < valid) y[(r0 + i) * ldy_row + j] = v;
    }
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kCanThreads, 1) can_head_kernel(CanArgs a, float* __restrict__ out) {
  extern __shared__ __align__(16) float sm[];
  const int D = a.D, M = a.w.n_modals;
  const int in_rows = max(a.c_max, D);
  float* s_in = sm;                                  // [max(C_max, D)][kCanRows]: z_i, later fc1's output
  float* s_cat = s_in + (size_t)in_rows * kCanRows;  // [D][kCanRows]
  float* s_g = s_cat + (size_t)D * kCanRows;         // [D][kCanRows]: gate logits, then softmax(gate) * cat
  float* s_w = s_g + (size_t)D * kCanRows;           // [2][kCanKC][max N]
  __shared__ float s_red[kCanThreads / 32][kCanRows];

  const long long row0 = (long long)blockIdx.x * kCanRows;
  const long long valid = min((long long)kCanRows, a.rows - row0);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  for (int m = 0; m < M; ++m) {
    const int C = a.w.dim[m];
    const float* f = a.feat[m];
    for (int i = threadIdx.x; i < C * kCanRows; i += kCanThreads) {
      const int r = i % kCanRows, k = i / kCanRows;
      s_in[i] = r < valid ? __ldg(f + (row0 + r) * a.ld[m] + k) : 0.f;
    }
    __syncthreads();
    tile_linear(a.w.attn_w[m], a.w.attn_b[m], kCanAttn, C, s_in, s_cat + (size_t)m * kCanAttn * kCanRows, 0, valid, 0,
                s_w);
  }
  tile_linear(a.w.gate_w, a.w.gate_b, D, D, s_cat, s_g, 0, valid, 0, s_w);

  // softmax over the D gate logits of each row: lane = row, warp w reduces features [w * D / 8, (w + 1) * D / 8) in
  // ascending order, the eight partials are combined in warp order (D is a multiple of 128)
  const int span = D / (kCanThreads / 32), k_lo = warp * span;
  float mx = -INFINITY;
  for (int k = k_lo; k < k_lo + span; ++k) mx = fmaxf(mx, s_g[k * kCanRows + lane]);
  s_red[warp][lane] = mx;
  __syncthreads();
  mx = s_red[0][lane];
  for (int w = 1; w < kCanThreads / 32; ++w) mx = fmaxf(mx, s_red[w][lane]);
  float s = 0.f;
  for (int k = k_lo; k < k_lo + span; ++k) s += expf(s_g[k * kCanRows + lane] - mx);
  __syncthreads();                                   // every warp has read the maxima
  s_red[warp][lane] = s;
  __syncthreads();
  s = 0.f;
  for (int w = 0; w < kCanThreads / 32; ++w) s += s_red[w][lane];
  const float inv = 1.f / s;
  for (int k = k_lo; k < k_lo + span; ++k) {
    const int i = k * kCanRows + lane;
    s_g[i] = expf(s_g[i] - mx) * inv * s_cat[i];
  }
  __syncthreads();

  tile_linear(a.w.fc1_w, a.w.fc1_b, D, D, s_g, s_in, 0, valid, 1, s_w);
  tile_linear(a.w.fc2_w, a.w.fc2_b, a.w.n_out, D, s_in, out + row0 * a.w.n_out, a.w.n_out, valid, a.apply_tanh ? 2 : 0,
              s_w);
}

static size_t can_smem_bytes(int D, int c_max) {
  return ((size_t)(std::max(c_max, D) + 2 * D) * kCanRows + 2 * (size_t)kCanKC * std::max(D, kCanAttn)) * sizeof(float);
}

}  // namespace cer

extern "C" int cer_can_head_forward(const cer_can_head_weights* w, const float* const* feats, const int32_t* ld,
                                    int64_t rows, int32_t apply_tanh, float* out, void* stream) {
  using namespace cer;
  if (!w || !feats || !ld || !out || rows < 0 || (apply_tanh != 0 && apply_tanh != 1))
    return set_error(CER_ERR_INVALID, "cer_can_head_forward: bad argument");
  const int M = w->n_modals;
  if (M < 1 || M > CER_MAX_MODALS) return set_error(CER_ERR_INVALID, "cer_can_head_forward: n_modals must be 1..4");
  if (w->n_out < 1 || w->n_out > kCanMaxOut) return set_error(CER_ERR_INVALID, "cer_can_head_forward: n_out must be 1..64");
  CanArgs a{};
  a.w = *w;
  a.rows = rows;
  a.D = kCanAttn * M;
  a.apply_tanh = apply_tanh;
  for (int m = 0; m < M; ++m) {
    if (w->dim[m] < 1 || w->dim[m] > kCanMaxDim)
      return set_error(CER_ERR_INVALID, "cer_can_head_forward: every modality needs 1..512 channels");
    if (!w->attn_w[m] || !w->attn_b[m] || !feats[m] || ld[m] < w->dim[m])
      return set_error(CER_ERR_INVALID, "cer_can_head_forward: null modality input / weight or row pitch below its channels");
    a.feat[m] = feats[m];
    a.ld[m] = ld[m];
    a.c_max = std::max(a.c_max, (int)w->dim[m]);
  }
  if (!w->gate_w || !w->gate_b || !w->fc1_w || !w->fc1_b || !w->fc2_w || !w->fc2_b)
    return set_error(CER_ERR_INVALID, "cer_can_head_forward: null weight");
  if (rows == 0) return CER_OK;
  const long long tiles = (rows + kCanRows - 1) / kCanRows;
  if (tiles > 0x7fffffffLL) return set_error(CER_ERR_INVALID, "cer_can_head_forward: too many rows");
  const size_t smem = can_smem_bytes(a.D, a.c_max);
  static unsigned long long configured = 0;
  if (first_use_on_device(&configured))
    CER_CUDA(cudaFuncSetAttribute(can_head_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)can_smem_bytes(kCanMaxDim, kCanMaxDim)));
  set_head_variant("can_head_kernel");
  can_head_kernel<<<(unsigned)tiles, kCanThreads, smem, static_cast<cudaStream_t>(stream)>>>(a, out);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}
