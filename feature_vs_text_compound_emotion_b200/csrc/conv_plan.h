// Host-side plan pieces of the tcgen05 implicit-GEMM convolution shared by the IR-50 and VGGish
// plans: geometry -> tensor maps + kernel parameters, and the launcher that picks the kernel variant.
// Definitions live in ir50.cu (the only TU that instantiates the conv kernels).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include "conv_igemm.cuh"

namespace cer {

struct ConvOp {
  ConvKernelParams kp;
  CUtensorMap tmap_b_half;   // weights with a BN/2-row box: the CTA-pair variant loads half a B tile per CTA
  int bn;          // 64 / 128 / 256
  int hw_out;      // output pixels per frame
  CUtensorMap tmap_halo;     // tiled 4-D map with an 18 x 10 pixel box (conv_halo_kernel); valid iff halo_ok
  int halo_ok;               // 3x3 / stride 1 / pad 1, Cin = 64, Cout in {64, 128}, W % 8 == 0
  CUtensorMap tmap_strip;    // tiled 4-D map with an 8-row x 10-pixel box (conv_strip_kernel); valid iff strip_ok
  int strip_ok;              // halo_ok, Cout = 64, H % 8 == 0, no fused pooling
};

struct ConvGeom {
  const void* src; int H, W, Cin, ksize, stride, pad;
  const void* src2; int H2, W2, Cin2, stride2;       // fused shortcut operand (Cin2 = 0: none)
  const void* weight; const float* bias; int bias_classes; const float* alpha;
  const __nv_bfloat16* res; void* dst; int Cout; int out_fp32;
  int pool;        // 1: fuse MaxPool2d(2,2) into the epilogue (dst is the pooled tensor); see conv_can_pool()
  int wld;         // elements per weight row (0: the conv's K); a conv over a column slice of a wider weight matrix
};

int load_driver_entry_points();
// can a 3x3/s1/p1 conv over an H x W map with these channels fuse the 2x2 max-pool into its epilogue?
bool conv_can_pool(int H, int W, int Cin, int Cout);
// n_cap: frames the activation allocation holds (tensor-map N extent)
// host_tables: also copy the per-channel epilogue constants into the kernel parameters (synchronous D2H: plan creation only)
int build_conv_op(ConvOp* op, const ConvGeom& g, int n_cap, bool host_tables = false);
// out_wp != 0: store the output as a padded raster of row pitch out_wp = Wout + 1 (im2col kernels only; conv_raster.cuh)
int launch_conv(const ConvOp& op, int frames, int num_sms, cudaStream_t st, int out_wp = 0);
// name of the kernel instantiation launch_conv picks for `op` at `frames` frames / launched last on this thread
const char* conv_variant_name(const ConvOp& op, int frames, int num_sms);
const char* conv_last_variant();

}  // namespace cer
