// Five-point face alignment on the device: full frames -> the aligned uint8 face crops the video stream takes.
// C-ABI: cer_face_fit, cer_face_warp (include/cer_b200.h).
// Reference: face.evoLVe's warp_and_crop_face (align_trans.py) with reflective=True, i.e.
// matlab_cp2tform.get_similarity_transform_for_cv2 followed by cv2.warpAffine(img, M, (S, S)), as the offline
// pipeline's dlib / retinaface alignment runs it (SURVEY §2.1 row 19).
//
// face_fit_kernel: one thread per face, fp64.  The 4 x 4 normal equations of the similarity least squares have a
// closed form after centring, so no general solver is needed.  The cv2 inversion is restated with explicit
// round-to-nearest operations in cv::warpAffine's own order, so the inverse matrix is bit-identical with the one
// OpenCV derives from the same forward matrix.
//
// face_warp_kernel: OpenCV's fixed-point INTER_LINEAR / BORDER_CONSTANT 0 (imgwarp.cpp WarpAffineInvoker +
// remapBilinear).  One CTA per (face, band of output rows): every thread computes whole pixels into shared memory,
// then the band, which is contiguous in the output, leaves with 16-byte stores.  Taps are byte loads through L1.
#include <cuda_runtime.h>
#include <cstdint>

#include "../../include/cer_b200.h"
#include "common.h"

namespace cer {

constexpr int kWarpThreads = 256;
constexpr int kBandPixels = 2048;   // output pixels per CTA: rows_per_band = max(1, kBandPixels / S)

struct FaceRef {
  double x[5], y[5];
};

// findNonreflectiveSimilarity(uv = src, xy = ref): least squares of u = a x + b y + tx, v = -b x + a y + ty, returned
// as the 2 x 3 forward matrix (source -> reference) cv2 receives: rows of inv(Tinv)[:, 0:2].T.
__device__ __forceinline__ void nonreflective(const double* u, const double* v, const double* x, const double* y,
                                              double* M) {
  double xm = 0, ym = 0, um = 0, vm = 0;
#pragma unroll
  for (int i = 0; i < 5; ++i) { xm += x[i]; ym += y[i]; um += u[i]; vm += v[i]; }
  xm /= 5; ym /= 5; um /= 5; vm /= 5;
  double sxx = 0, sa = 0, sb = 0;
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    const double xc = x[i] - xm, yc = y[i] - ym, uc = u[i] - um, vc = v[i] - vm;
    sxx += xc * xc + yc * yc;
    sa += xc * uc + yc * vc;
    sb += yc * uc - xc * vc;
  }
  const double a = sa / sxx, b = sb / sxx;
  const double tx = um - a * xm - b * ym, ty = vm + b * xm - a * ym;
  const double det = a * a + b * b;
  M[0] = a / det;  M[1] = -b / det; M[2] = -(a * tx - b * ty) / det;
  M[3] = b / det;  M[4] = a / det;  M[5] = -(b * tx + a * ty) / det;
}

__device__ __forceinline__ double residual(const double* M, const double* u, const double* v, const double* x,
                                           const double* y) {
  double s = 0;
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    const double dx = u[i] * M[0] + v[i] * M[1] + M[2] - x[i];
    const double dy = u[i] * M[3] + v[i] * M[4] + M[5] - y[i];
    s += dx * dx + dy * dy;
  }
  return sqrt(s);
}

__global__ void __launch_bounds__(128) face_fit_kernel(const float* __restrict__ lm, long long n, FaceRef ref,
                                                       double* __restrict__ fwd, double* __restrict__ inv) {
  const long long f = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (f >= n) return;
  double u[5], v[5], xr[5];
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    u[i] = lm[f * 10 + 2 * i];
    v[i] = lm[f * 10 + 2 * i + 1];
    xr[i] = -ref.x[i];
  }
  double M1[6], M2[6];
  nonreflective(u, v, ref.x, ref.y, M1);
  nonreflective(u, v, xr, ref.y, M2);   // fit to the mirrored reference, then compose with the reflection
  M2[0] = -M2[0]; M2[1] = -M2[1]; M2[2] = -M2[2];
  const double* M = residual(M1, u, v, ref.x, ref.y) <= residual(M2, u, v, ref.x, ref.y) ? M1 : M2;
  // cv::warpAffine's inversion of the matrix it is given, operation for operation
  double D = __dsub_rn(__dmul_rn(M[0], M[4]), __dmul_rn(M[1], M[3]));
  D = D != 0.0 ? __ddiv_rn(1.0, D) : 0.0;
  const double A11 = __dmul_rn(M[4], D), A22 = __dmul_rn(M[0], D);
  const double A12 = __dmul_rn(M[1], -D), A21 = __dmul_rn(M[3], -D);
  const double b1 = __dsub_rn(__dmul_rn(-A11, M[2]), __dmul_rn(A12, M[5]));
  const double b2 = __dsub_rn(__dmul_rn(-A21, M[2]), __dmul_rn(A22, M[5]));
  double* F = fwd + f * 6;
  double* I = inv + f * 6;
#pragma unroll
  for (int k = 0; k < 6; ++k) F[k] = M[k];
  I[0] = A11; I[1] = A12; I[2] = b1;
  I[3] = A21; I[4] = A22; I[5] = b2;
}

// OpenCV's source position of output pixel (x, y), in 1/32 px: cvRound(...) is round-half-even, as __double2int_rn.
__device__ __forceinline__ int fixed_coord(double a_x, double a_y, double b, int x, int y) {
  const int row = __double2int_rn(__dmul_rn(__dadd_rn(__dmul_rn(a_y, (double)y), b), 1024.0)) + 16;
  const int step = __double2int_rn(__dmul_rn(__dmul_rn(a_x, (double)x), 1024.0));
  return (row + step) >> 5;
}

__global__ void __launch_bounds__(kWarpThreads) face_warp_kernel(const uint8_t* __restrict__ frames, long long n_frames,
                                                                 int h, int w, const long long* __restrict__ frame_index,
                                                                 const double* __restrict__ inv, int S, int band_rows,
                                                                 int n_bands, uint8_t* __restrict__ out) {
  __shared__ __align__(16) uint8_t s_band[kBandPixels * 3 + 16];
  const long long face = blockIdx.x / n_bands;
  const int y0 = (int)(blockIdx.x - face * n_bands) * band_rows;
  const int rows = min(band_rows, S - y0);
  const double* A = inv + face * 6;
  const double A11 = A[0], A12 = A[1], A13 = A[2], A21 = A[3], A22 = A[4], A23 = A[5];
  const long long fi = frame_index[face];
  const bool in_range = fi >= 0 && fi < n_frames;     // an index outside the buffer reads nothing: a zero crop
  const uint8_t* img = frames + (in_range ? fi : 0) * ((long long)h * w * 3);
  uint8_t* dst = out + (face * S + y0) * (long long)S * 3;
  const int lead = (int)(reinterpret_cast<uintptr_t>(dst) & 15);
  uint8_t* sb = s_band + lead;                         // sb[i] and dst[i] share their address mod 16
  const int n_px = rows * S;
  for (int i = threadIdx.x; i < n_px; i += kWarpThreads) {
    const int yy = i / S, x = i - yy * S, y = y0 + yy;
    const int X = fixed_coord(A11, A12, A13, x, y);
    const int Y = fixed_coord(A21, A22, A23, x, y);
    const int sx = min(max(X >> 5, -32768), 32767), fx = X & 31;   // saturate_cast<short>, as OpenCV's map
    const int sy = min(max(Y >> 5, -32768), 32767), fy = Y & 31;
    int acc0 = 0, acc1 = 0, acc2 = 0;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy) {
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        const int tx = sx + dx, ty = sy + dy;
        if (in_range && (unsigned)tx < (unsigned)w && (unsigned)ty < (unsigned)h) {
          // 15-bit weights: (1/32-px fractions) products are exact and sum to 32768
          const int wgt = (dy ? fy : 32 - fy) * (dx ? fx : 32 - fx) * 32;
          const uint8_t* p = img + ((long long)ty * w + tx) * 3;
          acc0 += __ldg(p) * wgt;
          acc1 += __ldg(p + 1) * wgt;
          acc2 += __ldg(p + 2) * wgt;
        }
      }
    }
    uint8_t* s = sb + i * 3;
    s[0] = (uint8_t)min((acc0 + (1 << 14)) >> 15, 255);
    s[1] = (uint8_t)min((acc1 + (1 << 14)) >> 15, 255);
    s[2] = (uint8_t)min((acc2 + (1 << 14)) >> 15, 255);
  }
  __syncthreads();
  const int total = n_px * 3;
  const int head = min(total, (16 - lead) & 15);
  const int n16 = (total - head) >> 4;
  if (threadIdx.x < head) dst[threadIdx.x] = sb[threadIdx.x];
  const uint4* s4 = reinterpret_cast<const uint4*>(sb + head);
  uint4* d4 = reinterpret_cast<uint4*>(dst + head);
  for (int i = threadIdx.x; i < n16; i += kWarpThreads) d4[i] = s4[i];
  for (int i = head + n16 * 16 + threadIdx.x; i < total; i += kWarpThreads) dst[i] = sb[i];
}

}  // namespace cer

using namespace cer;

extern "C" int cer_face_fit(const float* landmarks_dev, int64_t n, const double* reference_host, double* fwd_dev,
                            double* inv_dev, void* stream) {
  if (n < 0 || n > (1ll << 31) || (n > 0 && (!landmarks_dev || !fwd_dev || !inv_dev)) || !reference_host)
    return set_error(CER_ERR_INVALID, "cer_face_fit: bad argument (null pointer or n outside [0, 2^31])");
  FaceRef ref;
  double xm = 0, ym = 0;
  for (int i = 0; i < 5; ++i) {
    ref.x[i] = reference_host[2 * i];
    ref.y[i] = reference_host[2 * i + 1];
    if (!(ref.x[i] - ref.x[i] == 0.0 && ref.y[i] - ref.y[i] == 0.0))
      return set_error(CER_ERR_INVALID, "cer_face_fit: reference points must be finite");
    xm += ref.x[i] / 5;
    ym += ref.y[i] / 5;
  }
  double spread = 0;
  for (int i = 0; i < 5; ++i) spread += (ref.x[i] - xm) * (ref.x[i] - xm) + (ref.y[i] - ym) * (ref.y[i] - ym);
  if (!(spread > 0)) return set_error(CER_ERR_INVALID, "cer_face_fit: the reference points must not all coincide");
  if (n == 0) return CER_OK;
  face_fit_kernel<<<(unsigned)((n + 127) / 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(landmarks_dev, n, ref,
                                                                                            fwd_dev, inv_dev);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

extern "C" int cer_face_warp(const uint8_t* frames_dev, int64_t n_frames, int32_t h, int32_t w,
                             const int64_t* frame_index_dev, const double* inv_dev, int64_t n, int32_t crop,
                             uint8_t* out_dev, void* stream) {
  if (n < 0 || crop < 1 || crop > 1024 || h < 1 || h > 32767 || w < 1 || w > 32767 || n_frames < 0)
    return set_error(CER_ERR_INVALID, "cer_face_warp: shape outside the limits (crop 1..1024, h and w 1..32767)");
  if (n > 0 && (!frames_dev || !frame_index_dev || !inv_dev || !out_dev || n_frames == 0))
    return set_error(CER_ERR_INVALID, "cer_face_warp: bad argument (null pointer or no frames)");
  const int band_rows = crop >= kBandPixels ? 1 : min(crop, kBandPixels / crop);
  const int n_bands = (crop + band_rows - 1) / band_rows;
  if (n > ((1ll << 31) - 1) / n_bands) return set_error(CER_ERR_INVALID, "cer_face_warp: too many faces for one call");
  if (n == 0) return CER_OK;
  face_warp_kernel<<<(unsigned)(n * n_bands), kWarpThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      frames_dev, n_frames, h, w, reinterpret_cast<const long long*>(frame_index_dev), inv_dev, crop, band_rows,
      n_bands, out_dev);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}
