// Log-mel front end of the inline-VGGish modality on the device.  C-ABI: cer_logmel_forward,
// cer_frame_examples, and their streaming forms cer_stream_logmel, cer_stream_examples (include/cer_b200.h).
// Reference: abaw5_pre_processing/base/vggish/mel_features.py:92-236 (stft_magnitude, periodic_hann,
// spectrogram_to_mel_matrix, log_mel_spectrogram) and my_frame (:21-46) / vggish_input.py:37-82.
//
// The reference computes in float64 (numpy).  The whole front end is 0.44 MFLOP per 10 ms frame, so
// it is done in fp64 here as well (B200: ~40 TFLOP/s fp64, the cost is negligible next to VGGish's
// 1.7 GFLOP per example) and agrees with numpy to ~1e-12 before the final cast to fp32.
//   DFT by definition: X[k] = sum_n x[n] w[n] (cos, -sin)(2 pi k n / fft), twiddles from a table of
//   fft entries indexed (k*n) mod fft; |X| -> mel matrix [bins][mel] -> log(. + offset).
// One CTA per 4 STFT frames (each twiddle read feeds 4 frames); thread k owns spectrogram bin k,
// then one thread per (frame, mel band).
#include <cuda_runtime.h>
#include <cstdint>

#include "../../include/cer_b200.h"
#include "common.h"

namespace cer {

constexpr int kLmFrames = 4;      // STFT frames per CTA: every twiddle read from smem feeds 4 frames

// The log-mel rows f0 .. f0 + kLmFrames - 1 of one CTA, of which the first n_valid are real.  sample(q, n) is sample
// n of row f0 + q, row_out(q) the fp32 [n_mel] destination of row f0 + q.  Both the offline kernel and the
// streaming kernel run this body, so a row's fp64 arithmetic (and its fma order) does not depend on where its
// samples came from: it is bit-identical however the samples were split across calls.
template <class Sample, class RowOut>
__device__ __forceinline__ void logmel_rows(const Sample& sample, const RowOut& row_out, int n_valid,
                                            const double* __restrict__ tables, int win, int fft, int n_mel,
                                            double log_offset) {
  extern __shared__ __align__(16) double sm_d[];
  double* s_x = sm_d;                            // [win][kLmFrames] windowed samples, frame-minor
  double* s_cos = s_x + win * kLmFrames;         // [fft]
  double* s_sin = s_cos + fft;                   // [fft]
  double* s_mag = s_sin + fft;                   // [kLmFrames][fft/2 + 1]
  const int bins = fft / 2 + 1;
  const double* hann = tables;        // [win]
  const double* tcos = tables + win;  // [fft]
  const double* tsin = tcos + fft;    // [fft]
  const double* mel = tsin + fft;     // [bins][n_mel]
  for (int i = threadIdx.x; i < win * kLmFrames; i += blockDim.x) {
    const int n = i / kLmFrames, q = i - n * kLmFrames;
    s_x[i] = q < n_valid ? (double)sample(q, n) * hann[n] : 0.0;
  }
  for (int i = threadIdx.x; i < fft; i += blockDim.x) { s_cos[i] = tcos[i]; s_sin[i] = tsin[i]; }
  __syncthreads();
  for (int k = threadIdx.x; k < bins; k += blockDim.x) {
    double re[kLmFrames], im[kLmFrames];
#pragma unroll
    for (int q = 0; q < kLmFrames; ++q) { re[q] = 0.0; im[q] = 0.0; }
    int idx = 0;                                   // (k * n) mod fft, fft is a power of two
    for (int n = 0; n < win; ++n) {
      const double c = s_cos[idx], sn = s_sin[idx];
      const double2 x01 = *reinterpret_cast<const double2*>(&s_x[n * kLmFrames]);
      const double2 x23 = *reinterpret_cast<const double2*>(&s_x[n * kLmFrames + 2]);
      re[0] = fma(x01.x, c, re[0]); im[0] = fma(x01.x, sn, im[0]);
      re[1] = fma(x01.y, c, re[1]); im[1] = fma(x01.y, sn, im[1]);
      re[2] = fma(x23.x, c, re[2]); im[2] = fma(x23.x, sn, im[2]);
      re[3] = fma(x23.y, c, re[3]); im[3] = fma(x23.y, sn, im[3]);
      idx = (idx + k) & (fft - 1);
    }
#pragma unroll
    for (int q = 0; q < kLmFrames; ++q) s_mag[q * bins + k] = sqrt(re[q] * re[q] + im[q] * im[q]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n_mel * kLmFrames; i += blockDim.x) {
    const int q = i / n_mel, j = i - q * n_mel;
    if (q >= n_valid) continue;
    double acc = 0.0;
    const double* mg = s_mag + q * bins;
    for (int k = 0; k < bins; ++k) acc = fma(mg[k], mel[(long long)k * n_mel + j], acc);
    row_out(q)[j] = (float)log(acc + log_offset);
  }
}

__global__ void __launch_bounds__(288) logmel_kernel(const float* __restrict__ wave, long long n_samples,
                                                     const double* __restrict__ tables, int win, int hop, int fft, int n_mel,
                                                     double log_offset, float* __restrict__ out, int n_frames) {
  const int f0 = blockIdx.x * kLmFrames;
  logmel_rows([&](int q, int n) { return wave[(long long)(f0 + q) * hop + n]; },
              [&](int q) { return out + (long long)(f0 + q) * n_mel; }, min(kLmFrames, n_frames - f0), tables, win, fft,
              n_mel, log_offset);
}

// Streaming: blockIdx.y is one stream's work entry, blockIdx.x a group of kLmFrames of its new rows.  Sample p of
// the stream (p < a0: received earlier) comes from its tail, which holds samples a0 - tail_len .. a0 - 1; p >= a0
// from the packed new samples.  Row f goes to ring row f % ring_rows.
__global__ void __launch_bounds__(288) stream_logmel_kernel(const cer_stream_audio_entry* __restrict__ tab,
                                                            const float* __restrict__ samples,
                                                            const float* __restrict__ tails, int tail_len,
                                                            const double* __restrict__ tables, int win, int hop, int fft,
                                                            int n_mel, double log_offset, float* __restrict__ ring,
                                                            int ring_rows) {
  const cer_stream_audio_entry e = tab[blockIdx.y];
  // more new rows than the ring holds: only the last ring_rows are kept (and computed), as stream_retain_kernel does
  const int g0 = max(0, e.n_rows - ring_rows) + blockIdx.x * kLmFrames;
  if (g0 >= e.n_rows) return;                    // uniform over the CTA, before any barrier
  const long long f0 = (long long)e.first_row + g0;
  const float* tail = tails + (size_t)e.slot * tail_len;
  const long long tail0 = e.a0 - tail_len;
  float* slot_ring = ring + (size_t)e.slot * ring_rows * n_mel;
  logmel_rows(
      [&](int q, int n) {
        const long long p = (f0 + q) * hop + n;
        return p >= e.a0 ? samples[e.src_off + (p - e.a0)] : tail[p - tail0];
      },
      [&](int q) { return slot_ring + (size_t)((f0 + q) % ring_rows) * n_mel; }, min(kLmFrames, e.n_rows - g0), tables,
      win, fft, n_mel, log_offset);
}

// The tail after the push: samples a0 + n_new - tail_len .. a0 + n_new - 1 (zeros before the stream's sample 0).
// One CTA per entry; staged through shared memory, so reading the old tail and writing the new one do not race.
__global__ void __launch_bounds__(256) stream_tail_kernel(const cer_stream_audio_entry* __restrict__ tab,
                                                          const float* __restrict__ samples, float* __restrict__ tails,
                                                          int tail_len) {
  extern __shared__ float s_tail[];
  const cer_stream_audio_entry e = tab[blockIdx.x];
  float* tail = tails + (size_t)e.slot * tail_len;
  const long long a1 = e.a0 + e.n_new;
  for (int i = threadIdx.x; i < tail_len; i += blockDim.x) {
    const long long p = a1 - tail_len + i;
    s_tail[i] = p < 0 ? 0.f : p >= e.a0 ? samples[e.src_off + (p - e.a0)] : tail[p - (e.a0 - tail_len)];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < tail_len; i += blockDim.x) tail[i] = s_tail[i];
}

// out[dst][t][:] = ring[slot][(start + t) % ring_rows][:]: the ring form of frame_examples_kernel.
__global__ void stream_examples_kernel(const float* __restrict__ ring, int ring_rows, const int* __restrict__ entries,
                                       int n_examples, int frames_per_example, int n_mel, float* __restrict__ out) {
  const long long per = (long long)frames_per_example * n_mel;
  const long long total = (long long)n_examples * per;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int e = (int)(i / per);
    const int r = (int)(i - (long long)e * per);
    const int t = r / n_mel, j = r - t * n_mel;
    const int slot = entries[3 * e], start = entries[3 * e + 1], dst = entries[3 * e + 2];
    out[(long long)dst * per + r] = ring[((size_t)slot * ring_rows + (start + t) % ring_rows) * n_mel + j];
  }
}

// examples[e][t][:] = logmel[starts[e] + t][:]   (my_frame, mel_features.py:21-46)
__global__ void frame_examples_kernel(const float* __restrict__ logmel, const int* __restrict__ starts, int n_examples,
                                      int frames_per_example, int n_mel, float* __restrict__ out) {
  const long long per = (long long)frames_per_example * n_mel;
  const long long total = (long long)n_examples * per;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int e = (int)(i / per);
    const long long r = i - (long long)e * per;
    out[i] = logmel[(long long)starts[e] * n_mel + r];
  }
}

}  // namespace cer

using namespace cer;

extern "C" int64_t cer_logmel_num_frames(int64_t n_samples, int32_t win, int32_t hop) {
  if (n_samples < win || win <= 0 || hop <= 0) return 0;
  return 1 + (n_samples - win) / hop;
}

extern "C" int cer_logmel_forward(const float* wave_dev, int64_t n_samples, const double* tables_dev, int32_t win, int32_t hop,
                                  int32_t fft, int32_t n_mel, double log_offset, float* logmel_out_dev, void* stream) {
  if (!wave_dev || !tables_dev || !logmel_out_dev || win <= 0 || hop <= 0 || fft < win || (fft & (fft - 1)) || n_mel <= 0 ||
      fft > 4096)
    return set_error(CER_ERR_INVALID, "cer_logmel_forward: bad argument (fft must be a power of two >= win)");
  const int64_t n_frames = cer_logmel_num_frames(n_samples, win, hop);
  if (n_frames <= 0) return CER_OK;
  if (n_frames > (1ll << 30)) return set_error(CER_ERR_INVALID, "cer_logmel_forward: too many frames");
  const size_t smem = (size_t)(win * kLmFrames + 2 * fft + kLmFrames * (fft / 2 + 1)) * sizeof(double);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(logmel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return set_error(CER_ERR_CUDA, std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e));
  }
  logmel_kernel<<<(int)((n_frames + kLmFrames - 1) / kLmFrames), 288, smem, static_cast<cudaStream_t>(stream)>>>(wave_dev, n_samples, tables_dev, win, hop, fft,
                                                                                n_mel, log_offset, logmel_out_dev, (int)n_frames);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

extern "C" int cer_frame_examples(const float* logmel_dev, const int32_t* starts_dev, int32_t n_examples,
                                  int32_t frames_per_example, int32_t n_mel, float* out_dev, void* stream) {
  if (!logmel_dev || !starts_dev || !out_dev || n_examples < 0 || frames_per_example <= 0 || n_mel <= 0)
    return set_error(CER_ERR_INVALID, "cer_frame_examples: bad argument");
  if (n_examples == 0) return CER_OK;
  const long long total = (long long)n_examples * frames_per_example * n_mel;
  const int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  frame_examples_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(logmel_dev, starts_dev, n_examples,
                                                                               frames_per_example, n_mel, out_dev);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

extern "C" int cer_stream_logmel(const cer_stream_audio_entry* table_dev, int32_t n_entries, int32_t max_rows,
                                 const float* samples_dev, const double* tables_dev, int32_t win, int32_t hop, int32_t fft,
                                 int32_t n_mel, double log_offset, float* tails_dev, int32_t tail_len, float* ring_dev,
                                 int32_t ring_rows, void* stream) {
  if (!table_dev || !tables_dev || !tails_dev || !ring_dev || n_entries < 0 || n_entries > 65535 || max_rows < 0 ||
      win <= 0 || hop <= 0 || fft < win || (fft & (fft - 1)) || fft > 4096 || n_mel <= 0 || tail_len < win - 1 ||
      tail_len > 12 * 1024 || ring_rows <= 0)
    return set_error(CER_ERR_INVALID, "cer_stream_logmel: bad argument (needs tail_len >= win - 1, fft a power of two >= win)");
  if (n_entries == 0) return CER_OK;
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (max_rows > 0) {
    const size_t smem = (size_t)(win * kLmFrames + 2 * fft + kLmFrames * (fft / 2 + 1)) * sizeof(double);
    if (smem > 48 * 1024) {
      cudaError_t e = cudaFuncSetAttribute(stream_logmel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return set_error(CER_ERR_CUDA, std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e));
    }
    const int rows = max_rows < ring_rows ? max_rows : ring_rows;
    const dim3 grid((rows + kLmFrames - 1) / kLmFrames, n_entries);
    stream_logmel_kernel<<<grid, 288, smem, st>>>(table_dev, samples_dev, tails_dev, tail_len, tables_dev, win, hop, fft,
                                                  n_mel, log_offset, ring_dev, ring_rows);
    CER_CUDA(cudaGetLastError());
  }
  stream_tail_kernel<<<n_entries, 256, tail_len * sizeof(float), st>>>(table_dev, samples_dev, tails_dev, tail_len);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

extern "C" int cer_stream_examples(const float* ring_dev, int32_t ring_rows, const int32_t* entries_dev, int32_t n_examples,
                                   int32_t frames_per_example, int32_t n_mel, float* out_dev, void* stream) {
  if (!ring_dev || !entries_dev || !out_dev || ring_rows <= 0 || n_examples < 0 || frames_per_example <= 0 ||
      frames_per_example > ring_rows || n_mel <= 0)
    return set_error(CER_ERR_INVALID, "cer_stream_examples: bad argument");
  if (n_examples == 0) return CER_OK;
  const long long total = (long long)n_examples * frames_per_example * n_mel;
  const int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  stream_examples_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(ring_dev, ring_rows, entries_dev,
                                                                                n_examples, frames_per_example, n_mel,
                                                                                out_dev);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}
