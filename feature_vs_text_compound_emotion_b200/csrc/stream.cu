// Streaming LFAN head: per-stream state around the unchanged TCN and fusion kernels.
//
// A session advances n streams by c frames per step.  Each (stream, window) pair active in the step is one
// "entry" of a small table (cer_stream_entry, written by the host, copied once per step); entries are laid out
// [n][n_slots] with each stream's windows in start order and the unused ones flagged inactive, so every step is
// the same sequence of launches whatever phase each stream is in.
//
// Per TemporalBlock b (halo h = (k-1)*d, R = 2h ring rows) an entry's staged input is [R + c][C_in] rows of
// absolute frames o, o+1, ... with o = max(start, t_now - R):
//   * an old window (start <= t_now - R): the R frames before the chunk come from the ring, so conv1 is exact
//     from row h on and conv2 (which reads h1 rows t-h..t) is exact on the last c rows;
//   * a young window (start > t_now - R): row 0 is the window's first frame, so the TMA zero fill before row 0
//     is exactly the offline kernel's causal padding, for conv1 *and* conv2 (h1 rows before the window's start
//     are padding, not LReLU(b1)).
// The TC kernel then runs on [entries][R + c][C_in] unchanged; the next block stages from its output rows.
// The ring keeps the last R rows of each block's input per (stream, window slot), in two halves: a step reads
// half `parity` and writes the other, so no thread overwrites a row another thread still reads.
#include <cuda_runtime.h>
#include <cstdint>

#include "../../include/cer_b200.h"
#include "common.h"

namespace cer {

constexpr int kStreamThreads = 256;

__device__ __forceinline__ int stage_origin(const cer_stream_entry& e, int ring_rows) {
  return max(e.start, e.t_now - ring_rows);
}

__global__ void __launch_bounds__(kStreamThreads) stream_stage_kernel(
    const cer_stream_entry* __restrict__ tab, int n_entries, int n_slots, int chunk, int ring_rows, int c_pad,
    const float* __restrict__ src, int src_dim, int src_len, int src_ring_rows, float* __restrict__ ring,
    float* __restrict__ staged) {
  const int L = ring_rows + chunk;
  const long long total = (long long)n_entries * L * c_pad;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int ci = (int)(idx % c_pad);
    const long long er = idx / c_pad;
    const int r = (int)(er % L);
    const int ei = (int)(er / L);
    const cer_stream_entry e = tab[ei];
    float v = 0.f;
    if (e.active) {
      const int o = stage_origin(e, ring_rows);
      const int f = o + r;
      const int end = e.t_now + chunk;
      if (f < end) {
        float* rbase = ring + ((size_t)(e.sid * n_slots + e.slot) * 2) * ring_rows * c_pad;
        if (f >= e.t_now) {
          if (ci < src_dim) {
            const size_t row = src_len == 0 ? (size_t)(ei / n_slots) * chunk + (f - e.t_now)
                                            : (size_t)ei * src_len + (f - stage_origin(e, src_ring_rows));
            v = src[row * src_dim + ci];
          }
        } else {
          v = rbase[((size_t)e.parity * ring_rows + f % ring_rows) * c_pad + ci];
        }
        if (ring_rows > 0 && f >= end - ring_rows)
          rbase[((size_t)(e.parity ^ 1) * ring_rows + f % ring_rows) * c_pad + ci] = v;
      }
    }
    staged[idx] = v;
  }
}

__global__ void __launch_bounds__(kStreamThreads) stream_gather_kernel(
    const cer_stream_entry* __restrict__ tab, int n_entries, int chunk, const float* __restrict__ src, int src_len,
    int src_ring_rows, int dim, float* __restrict__ dst) {
  const long long total = (long long)n_entries * chunk * dim;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % dim);
    const long long er = idx / dim;
    const int r = (int)(er % chunk);
    const int ei = (int)(er / chunk);
    const cer_stream_entry e = tab[ei];
    const int f = e.t_now + r;
    float v = 0.f;
    if (e.active && f >= e.start) v = src[((size_t)ei * src_len + (f - stage_origin(e, src_ring_rows))) * dim + c];
    dst[idx] = v;
  }
}

// The stitch arithmetic of stitch_kernel (fusion.cu): windows summed in start order from 0, then divided by the count.
__global__ void __launch_bounds__(kStreamThreads) stream_average_kernel(
    const cer_stream_entry* __restrict__ tab, int n_streams, int n_slots, int chunk, int window_length, int n_out,
    const float* __restrict__ win_logits, float* __restrict__ out, float* __restrict__ logit_ring, int n_lslots) {
  const long long total = (long long)n_streams * chunk * n_out;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % n_out);
    const long long ir = idx / n_out;
    const int r = (int)(ir % chunk);
    const int i = (int)(ir / chunk);
    float s = 0.f;
    int cnt = 0;
    for (int j = 0; j < n_slots; ++j) {
      const int ei = i * n_slots + j;
      const cer_stream_entry e = tab[ei];
      const int f = e.t_now + r;
      if (e.active && f >= e.start && f < e.start + window_length) {
        const float v = win_logits[((size_t)ei * chunk + r) * n_out + c];
        s += v;
        ++cnt;
        logit_ring[(((size_t)e.sid * n_lslots + e.lslot) * window_length + (f - e.start)) * n_out + c] = v;
      }
    }
    out[idx] = cnt > 0 ? s / cnt : 0.f;
  }
}

__global__ void __launch_bounds__(kStreamThreads) stream_retain_kernel(
    const cer_stream_entry* __restrict__ tab, int n_streams, int n_slots, int chunk, const float* __restrict__ src,
    int dim, int window_length, float* __restrict__ ring) {
  const long long total = (long long)n_streams * chunk * dim;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % dim);
    const long long ir = idx / dim;
    const int r = (int)(ir % chunk);
    const int i = (int)(ir / chunk);
    // a chunk longer than the ring keeps its last window_length rows: rows r and r + window_length share a ring row
    if (r < chunk - window_length) continue;
    const cer_stream_entry e = tab[(size_t)i * n_slots];
    ring[((size_t)e.sid * window_length + (e.t_now + r) % window_length) * dim + c] = src[idx];
  }
}

// A JMT / MT stream's history: the chunk rows of each entry (src [n_entries][chunk][dim], a gather's output) go to
// history [n_streams][max_frames][dim] at rows t_now .. t_now + chunk - 1.  Rows past max_frames and entries with a
// sid outside [0, n_streams) are dropped (the host refuses such pushes), so nothing outside the range is written.
__global__ void __launch_bounds__(kStreamThreads) stream_append_kernel(
    const cer_stream_entry* __restrict__ tab, int n_entries, int chunk, const float* __restrict__ src, int dim,
    int n_streams, int max_frames, float* __restrict__ history) {
  const long long total = (long long)n_entries * chunk * dim;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % dim);
    const long long er = idx / dim;
    const int r = (int)(er % chunk);
    const int ei = (int)(er / chunk);
    const cer_stream_entry e = tab[ei];
    const int f = e.t_now + r;
    if (e.active && e.sid >= 0 && e.sid < n_streams && f >= 0 && f < max_frames)
      history[((size_t)e.sid * max_frames + f) * dim + c] = src[idx];
  }
}

static int grid_for(long long total) {
  const long long blocks = (total + kStreamThreads - 1) / kStreamThreads;
  return (int)(blocks < 148LL * 16 ? (blocks > 0 ? blocks : 1) : 148LL * 16);
}

}  // namespace cer

extern "C" int cer_stream_stage(const cer_stream_entry* table_dev, int32_t n_entries, int32_t n_slots, int32_t chunk,
                                int32_t ring_rows, int32_t c_pad, const float* src_dev, int32_t src_dim, int32_t src_len,
                                int32_t src_ring_rows, float* ring_dev, float* staged_dev, void* stream) {
  using namespace cer;
  if (!table_dev || !src_dev || !staged_dev || (ring_rows > 0 && !ring_dev) || n_entries <= 0 || n_slots <= 0 ||
      chunk <= 0 || ring_rows < 0 || c_pad <= 0 || src_dim <= 0 || src_dim > c_pad || src_len < 0 ||
      src_ring_rows < 0 || (src_len > 0 && src_len != src_ring_rows + chunk))
    return set_error(CER_ERR_INVALID, "cer_stream_stage: bad argument");
  const long long total = (long long)n_entries * (ring_rows + chunk) * c_pad;
  stream_stage_kernel<<<grid_for(total), kStreamThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      table_dev, n_entries, n_slots, chunk, ring_rows, c_pad, src_dev, src_dim, src_len, src_ring_rows, ring_dev,
      staged_dev);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

extern "C" int cer_stream_gather(const cer_stream_entry* table_dev, int32_t n_entries, int32_t chunk, const float* src_dev,
                                 int32_t src_ring_rows, int32_t dim, float* dst_dev, void* stream) {
  using namespace cer;
  if (!table_dev || !src_dev || !dst_dev || n_entries <= 0 || chunk <= 0 || src_ring_rows < 0 || dim <= 0)
    return set_error(CER_ERR_INVALID, "cer_stream_gather: bad argument");
  const long long total = (long long)n_entries * chunk * dim;
  stream_gather_kernel<<<grid_for(total), kStreamThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      table_dev, n_entries, chunk, src_dev, src_ring_rows + chunk, src_ring_rows, dim, dst_dev);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

extern "C" int cer_stream_average(const cer_stream_entry* table_dev, int32_t n_streams, int32_t n_slots, int32_t chunk,
                                  int32_t window_length, int32_t n_out, const float* win_logits_dev, float* out_dev,
                                  float* logit_ring_dev, int32_t n_lslots, void* stream) {
  using namespace cer;
  if (!table_dev || !win_logits_dev || !out_dev || !logit_ring_dev || n_streams <= 0 || n_slots <= 0 || chunk <= 0 ||
      window_length <= 0 || n_out <= 0 || n_lslots < n_slots)
    return set_error(CER_ERR_INVALID, "cer_stream_average: bad argument");
  const long long total = (long long)n_streams * chunk * n_out;
  stream_average_kernel<<<grid_for(total), kStreamThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      table_dev, n_streams, n_slots, chunk, window_length, n_out, win_logits_dev, out_dev, logit_ring_dev, n_lslots);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

extern "C" int cer_stream_retain(const cer_stream_entry* table_dev, int32_t n_streams, int32_t n_slots, int32_t chunk,
                                 const float* src_dev, int32_t dim, int32_t window_length, float* ring_dev, void* stream) {
  using namespace cer;
  if (!table_dev || !src_dev || !ring_dev || n_streams <= 0 || n_slots <= 0 || chunk <= 0 || dim <= 0 ||
      window_length <= 0)
    return set_error(CER_ERR_INVALID, "cer_stream_retain: bad argument");
  const long long total = (long long)n_streams * chunk * dim;
  stream_retain_kernel<<<grid_for(total), kStreamThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      table_dev, n_streams, n_slots, chunk, src_dev, dim, window_length, ring_dev);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

extern "C" int cer_stream_append(const cer_stream_entry* table_dev, int32_t n_entries, int32_t chunk, const float* src_dev,
                                 int32_t dim, int32_t n_streams, int32_t max_frames, float* history_dev, void* stream) {
  using namespace cer;
  if (!table_dev || !src_dev || !history_dev || n_entries <= 0 || chunk <= 0 || dim <= 0 || n_streams <= 0 ||
      max_frames <= 0)
    return set_error(CER_ERR_INVALID, "cer_stream_append: bad argument");
  const long long total = (long long)n_entries * chunk * dim;
  stream_append_kernel<<<grid_for(total), kStreamThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      table_dev, n_entries, chunk, src_dev, dim, n_streams, max_frames, history_dev);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}
