// SE tail of the IR-SE units (SEModule, models/arcface_model.py:23-41): squeeze + excite, then gate * r + shortcut.
// Both kernels are HBM bound: the squeeze reads the unit's pre-gate output r once, the scale reads r and the
// shortcut and writes the gated output over r (4 x the unit output's bytes per unit in all).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>
#include <algorithm>

#include "common.h"
#include "se.h"

namespace cer {

static const int kSeThreads = 256;

__device__ __forceinline__ void se_unpack8(const uint4& v, float f[8]) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    f[2 * j] = __uint_as_float(w[j] << 16);
    f[2 * j + 1] = __uint_as_float(w[j] & 0xffff0000u);
  }
}

__device__ __forceinline__ uint32_t se_pack2(float a, float b) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}

// One CTA per frame.  Thread t sums channel group t % G (8 channels, one 16-byte vector) over pixels
// t / G, t / G + P, ... (G = C / 8 groups, P = 256 / G pixel lanes); the lanes are reduced through shared memory.
__global__ void __launch_bounds__(kSeThreads) se_squeeze_excite_kernel(const __nv_bfloat16* __restrict__ r,
                                                                       const float* __restrict__ fc1,
                                                                       const float* __restrict__ fc2,
                                                                       float* __restrict__ gate, int hw, int C, int hidden) {
  __shared__ float part[kSeThreads * 8];
  __shared__ float mean[512];
  __shared__ float hid[64];
  const int n = blockIdx.x, tid = threadIdx.x;
  const int G = C >> 3, P = kSeThreads / G;
  const int g = tid % G, lane_px = tid / G;
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  const uint4* src = reinterpret_cast<const uint4*>(r + static_cast<size_t>(n) * hw * C) + g;
#pragma unroll 4
  for (int px = lane_px; px < hw; px += P) {
    float f[8];
    se_unpack8(__ldg(src + static_cast<size_t>(px) * G), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] += f[j];
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) part[lane_px * C + g * 8 + j] = acc[j];
  __syncthreads();
  const float inv_hw = 1.f / static_cast<float>(hw);
  for (int c = tid; c < C; c += kSeThreads) {
    float s = 0.f;
    for (int l = 0; l < P; ++l) s += part[l * C + c];
    mean[c] = s * inv_hw;
  }
  __syncthreads();
  const int warp = tid >> 5, lane = tid & 31;
  for (int j = warp; j < hidden; j += kSeThreads / 32) {
    const float* w = fc1 + static_cast<size_t>(j) * C;
    float s = 0.f;
    for (int c = lane; c < C; c += 32) s = fmaf(__ldg(w + c), mean[c], s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) hid[j] = fmaxf(s, 0.f);
  }
  __syncthreads();
  for (int c = tid; c < C; c += kSeThreads) {
    const float* w = fc2 + static_cast<size_t>(c) * hidden;
    float z = 0.f;
    for (int j = 0; j < hidden; ++j) z = fmaf(__ldg(w + j), hid[j], z);
    gate[static_cast<size_t>(n) * C + c] = 1.f / (1.f + expf(-z));
  }
}

// One thread per 16-byte vector of r (8 channels of one pixel), grid-stride.
__global__ void __launch_bounds__(kSeThreads) se_scale_shortcut_kernel(__nv_bfloat16* __restrict__ r,
                                                                       const float* __restrict__ gate,
                                                                       const __nv_bfloat16* __restrict__ sc, int frames,
                                                                       int Ho, int Wo, int C, int sc_h, int sc_w,
                                                                       int sc_stride) {
  const int G = C >> 3;
  const int hwo = Ho * Wo;
  const long long total = static_cast<long long>(frames) * hwo * G;
  for (long long v = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; v < total;
       v += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long pix = v / G;
    const int g = static_cast<int>(v - pix * G);
    const int n = static_cast<int>(pix / hwo);
    const int rem = static_cast<int>(pix - static_cast<long long>(n) * hwo);
    const int y = rem / Wo, x = rem - y * Wo;
    const size_t sc_off = ((static_cast<size_t>(n) * sc_h + y * sc_stride) * sc_w + x * sc_stride) * C + g * 8;
    uint4* rp = reinterpret_cast<uint4*>(r) + v;
    float fr[8], fs[8];
    se_unpack8(*rp, fr);
    se_unpack8(__ldg(reinterpret_cast<const uint4*>(sc + sc_off)), fs);
    const float4* gp = reinterpret_cast<const float4*>(gate + static_cast<size_t>(n) * C + g * 8);
    const float4 g0 = __ldg(gp), g1 = __ldg(gp + 1);
    const float gv[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
    float o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = fmaf(fr[j], gv[j], fs[j]);
    *rp = make_uint4(se_pack2(o[0], o[1]), se_pack2(o[2], o[3]), se_pack2(o[4], o[5]), se_pack2(o[6], o[7]));
  }
}

int launch_se_squeeze(const __nv_bfloat16* r, const float* fc1, const float* fc2, float* gate, int frames, int hw, int C,
                      int hidden, cudaStream_t st) {
  if (frames <= 0) return CER_OK;
  se_squeeze_excite_kernel<<<frames, kSeThreads, 0, st>>>(r, fc1, fc2, gate, hw, C, hidden);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

int launch_se_scale(__nv_bfloat16* r, const float* gate, const __nv_bfloat16* sc, int frames, int Ho, int Wo, int C,
                    int sc_h, int sc_w, int sc_stride, int num_sms, cudaStream_t st) {
  if (frames <= 0) return CER_OK;
  const long long vecs = static_cast<long long>(frames) * Ho * Wo * (C / 8);
  const int blocks = static_cast<int>(std::min<long long>((vecs + kSeThreads - 1) / kSeThreads, 8LL * num_sms));
  se_scale_shortcut_kernel<<<blocks, kSeThreads, 0, st>>>(r, gate, sc, frames, Ho, Wo, C, sc_h, sc_w, sc_stride);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

}  // namespace cer
