// Squeeze-and-excitation tail of an IR-SE residual unit (se.cu), launched by the IR plan (ir50.cu).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>

namespace cer {

// gate[n][c] = sigmoid(fc2 . relu(fc1 . mean_hw(r[n, :, :, c]))), fp32; r bf16 NHWC [frames][hw][C].
// fc1: fp32 [hidden][C], fc2: fp32 [C][hidden].  Needs C % 8 == 0, 256 % (C / 8) == 0, C <= 512, hidden <= 64.
int launch_se_squeeze(const __nv_bfloat16* r, const float* fc1, const float* fc2, float* gate, int frames, int hw, int C,
                      int hidden, cudaStream_t st);

// r[n, y, x, c] = bf16(r[n, y, x, c] * gate[n][c] + sc[n, s*y, s*x, c]) in place, r: [frames][Ho][Wo][C],
// sc: [frames][sc_h][sc_w][C] (the unit input for an identity shortcut, the projection output with s = 1).
int launch_se_scale(__nv_bfloat16* r, const float* gate, const __nv_bfloat16* sc, int frames, int Ho, int Wo, int C,
                    int sc_h, int sc_w, int sc_stride, int num_sms, cudaStream_t st);

}  // namespace cer
