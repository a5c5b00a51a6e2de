// Microbenchmark of the two halves of the conv epilogue, on every SM at once (148 CTAs, one per SM):
//   ld:    tcgen05.ld 32x32b.x16 / .x32 / .x64 throughput per SM with 8 or 16 warps reading (warp w reads its
//          lane quarter w % 4, as in the conv kernels); bytes per cycle per SM.
//   store: a 128 x 128 bf16 output tile (256 B per pixel row) written by 16 warps of 32 columns each, like the
//          N = 128 epilogue, in two patterns:
//            lane  = one pixel row, 4 x STG.128 per 32 columns (each instruction touches 32 rows x 16 B);
//            xpose = a 4 x 4 uint4 transpose inside groups of four lanes (16 SHFL), after which each STG.128 covers
//                    8 rows x 64 B, i.e. whole 32 B sectors;
//            v8    = one pixel row per lane, 2 x STG.256 per 32 columns (whole sectors, no lane exchange).
//          The output (148 x 64 tiles x 32 KB = 310 MB) is larger than L2, so the stores drain to HBM.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o tools/epilogue_probe tools/epilogue_probe.cu
#include <cuda.h>
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include "../feature_vs_text_compound_emotion_b200/csrc/conv_igemm.cuh"

using namespace cer;

template <int X>
__device__ __forceinline__ void tmem_ld_x(uint32_t taddr, uint32_t (&v)[X]);
template <>
__device__ __forceinline__ void tmem_ld_x<16>(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
                 "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
               : "r"(taddr) : "memory");
}
template <>
__device__ __forceinline__ void tmem_ld_x<32>(uint32_t taddr, uint32_t (&v)[32]) { tmem_ld_32x32(taddr, v); }
template <>
__device__ __forceinline__ void tmem_ld_x<64>(uint32_t taddr, uint32_t (&v)[64]) {
  tmem_ld_32x32(taddr, *reinterpret_cast<uint32_t(*)[32]>(&v[0]));
  tmem_ld_32x32(taddr + 32, *reinterpret_cast<uint32_t(*)[32]>(&v[32]));
}

// .x64 is issued as two .x32 (one wait); a single .x64 asks for 64 output registers in one asm statement
template <int X>
__global__ void __launch_bounds__(512, 1) ld_probe(int iters, long long* cycles, uint32_t* sink) {
  __shared__ uint32_t tmem_slot;
  const int warp = threadIdx.x >> 5;
  const int nwarps = blockDim.x >> 5;
  if (warp == 0) { tmem_alloc(&tmem_slot, 512); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t base = tmem_slot + (static_cast<uint32_t>((warp & 3) * 32) << 16);
  const int col0 = (warp >> 2) * X;
  const int stride = (nwarps / 4) * X;
  uint32_t acc = 0;
  __syncthreads();
  const long long t0 = clock64();
  for (int i = 0; i < iters; ++i) {
    uint32_t v[X];
    tmem_ld_x<X>(base + ((col0 + i * stride) & 511), v);
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < X; ++j) acc ^= v[j];
  }
  __syncthreads();
  const long long t1 = clock64();
  if (threadIdx.x == 0) cycles[blockIdx.x] = t1 - t0;
  if (acc == 0x12345678u) sink[0] = acc;
  tc_fence_before();
  __syncthreads();
  if (warp == 0) { tc_fence_after(); tmem_dealloc(tmem_slot, 512); }
}

template <int MODE>
__global__ void __launch_bounds__(512, 1) store_probe(__nv_bfloat16* out, int tiles_per_cta, long long* cycles) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = (warp & 3) * 32 + lane;
  const int c0 = (warp >> 2) * 32;
  uint4 r[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) r[j] = make_uint4(row, c0 + j, blockIdx.x, 0x3f803f80u);
  __syncthreads();
  const long long t0 = clock64();
  for (int t = 0; t < tiles_per_cta; ++t) {
    const size_t tile = static_cast<size_t>(t) * gridDim.x + blockIdx.x;
    __nv_bfloat16* tp = out + tile * 128 * 128;
    if (MODE == 2) {
      __nv_bfloat16* op = tp + row * 128 + c0;
      st_global_256(op, r[0], r[1]);
      st_global_256(op + 16, r[2], r[3]);
    } else if (MODE == 0) {
      uint4* op = reinterpret_cast<uint4*>(tp + row * 128 + c0);
#pragma unroll
      for (int j = 0; j < 4; ++j) op[j] = r[j];
    } else {
      // 4 x 4 transpose of uint4 inside each group of four lanes: afterwards lane l holds segment l % 4 of the rows
      // 4 * (l / 4) + k, k = 0..3, of its group's four pixel rows
      uint4 s[4] = {r[0], r[1], r[2], r[3]};
      const int g = lane & 3;
#pragma unroll
      for (int k = 1; k < 4; ++k) {
        // exchange with lane ^ k: send the segment the partner owns, receive ours of its row
        // (register selects, not a run-time array index, so that s stays in registers)
        const int src = g ^ k;
        uint4 o = src == 0 ? s[0] : src == 1 ? s[1] : src == 2 ? s[2] : s[3];
        o.x = __shfl_xor_sync(0xffffffffu, o.x, k); o.y = __shfl_xor_sync(0xffffffffu, o.y, k);
        o.z = __shfl_xor_sync(0xffffffffu, o.z, k); o.w = __shfl_xor_sync(0xffffffffu, o.w, k);
#pragma unroll
        for (int m = 0; m < 4; ++m)
          if (m == src) s[m] = o;      // s[m] now holds segment g of row (group base + m)
      }
      const int grow = (warp & 3) * 32 + (lane & ~3);
#pragma unroll
      for (int k = 0; k < 4; ++k)
        reinterpret_cast<uint4*>(tp + (grow + k) * 128 + c0)[g] = s[k];
    }
  }
  __syncthreads();
  const long long t1 = clock64();
  if (threadIdx.x == 0) cycles[blockIdx.x] = t1 - t0;
}

static double mean_cycles(long long* d, int n) {
  long long h[1024];
  cudaMemcpy(h, d, n * sizeof(long long), cudaMemcpyDeviceToHost);
  double s = 0;
  for (int i = 0; i < n; ++i) s += h[i];
  return s / n;
}

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e), __FILE__, __LINE__); return 1; } } while (0)

template <int X>
static int run_ld(int sms, int warps, long long* cyc, uint32_t* sink) {
  const int iters = 4096;
  ld_probe<X><<<sms, warps * 32>>>(iters, cyc, sink);
  CK(cudaGetLastError());
  ld_probe<X><<<sms, warps * 32>>>(iters, cyc, sink);
  CK(cudaDeviceSynchronize());
  const double c = mean_cycles(cyc, sms);
  const double bytes = (double)warps * iters * 32 * X * 4;
  printf("tcgen05.ld 32x32b.x%-2d  %2d warps: %7.1f B/cycle/SM  (%.0f cycles per 32 KB column block of 128 lanes x 64 cols)\n",
         X, warps, bytes / c, c / (bytes / 32768.0));
  return 0;
}

template <int MODE>
static int run_store(int sms, __nv_bfloat16* out, int tiles_per_cta, long long* cyc) {
  store_probe<MODE><<<sms, 512>>>(out, tiles_per_cta, cyc);
  CK(cudaGetLastError());
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  cudaEventRecord(e0);
  store_probe<MODE><<<sms, 512>>>(out, tiles_per_cta, cyc);
  cudaEventRecord(e1);
  CK(cudaDeviceSynchronize());
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  const double c = mean_cycles(cyc, sms);
  const double bytes = (double)sms * tiles_per_cta * 128 * 128 * 2;
  printf("store %-5s: %6.1f cycles per 128x128 bf16 tile per SM, %.3f ms, %.2f TB/s\n", MODE == 0 ? "lane" : MODE == 1 ? "xpose" : "v8",
         c / tiles_per_cta, ms, bytes / (ms * 1e-3) / 1e12);
  return 0;
}

int main() {
  int sms = 0;
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, 0));
  printf("%s, %d SMs\n", prop.name, sms);
  long long* cyc;
  uint32_t* sink;
  CK(cudaMalloc(&cyc, 1024 * sizeof(long long)));
  CK(cudaMalloc(&sink, 4));
  for (int w : {8, 16}) {
    if (run_ld<16>(sms, w, cyc, sink) || run_ld<32>(sms, w, cyc, sink) || run_ld<64>(sms, w, cyc, sink)) return 1;
  }
  const int tiles_per_cta = 64;
  __nv_bfloat16* out;
  CK(cudaMalloc(&out, (size_t)sms * tiles_per_cta * 128 * 128 * 2));
  for (int rep = 0; rep < 2; ++rep)
    if (run_store<0>(sms, out, tiles_per_cta, cyc) || run_store<1>(sms, out, tiles_per_cta, cyc) ||
        run_store<2>(sms, out, tiles_per_cta, cyc)) return 1;
  cudaFree(out); cudaFree(cyc); cudaFree(sink);
  return 0;
}
