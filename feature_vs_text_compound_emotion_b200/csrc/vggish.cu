// VGGish audio backbone plan: conv1+ReLU+pool kernel, tcgen05 implicit-GEMM convs (bias + ReLU
// epilogue), 2x2 max-pool kernel, the three embedding FCs as 1x1 implicit GEMMs.
// C-ABI: cer_vggish_* in include/cer_b200.h.  Reference semantics: VGG / VGGish,
// models/backbone.py:16-66 (make_layers :43-53, embeddings :20-27, NHWC flatten :34-37).
#include <cuda_runtime.h>
#include <cuda.h>
#include <cuda_bf16.h>
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../include/cer_b200.h"
#include "common.h"
#include "conv_plan.h"

namespace cer {

// ------------------------------------------------------------------------------------------
// conv3x3(1 -> 64, pad 1) + bias + ReLU + MaxPool2d(2,2), fp32 [N,H,W] in -> bf16 NHWC
// [N,H/2,W/2,64] out.  K = 9 is not a tensor-core shape.  One thread = one pooled pixel, all 64
// channels: a 4x4 input patch in registers, weights [9][64] broadcast from shared memory.
// max and (+bias, ReLU) commute, so the four conv outputs are max-reduced before the bias.
// Reference: features.0-2, models/backbone.py:43-53.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) vgg_stem_pool_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                            const float* __restrict__ bias,
                                                            __nv_bfloat16* __restrict__ out, int n_patches, int H, int W) {
  __shared__ __align__(16) float ws[9 * 64];
  __shared__ __align__(16) float bs[64];
  for (int i = threadIdx.x; i < 9 * 64; i += blockDim.x) ws[i] = w[i];
  if (threadIdx.x < 64) bs[threadIdx.x] = bias[threadIdx.x];
  __syncthreads();
  const int Ho = H >> 1, Wo = W >> 1;
  const int hwo = Ho * Wo;
  const long long total = static_cast<long long>(n_patches) * hwo;
  for (long long pix = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; pix < total;
       pix += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int n = static_cast<int>(pix / hwo);
    const int rem = static_cast<int>(pix - static_cast<long long>(n) * hwo);
    const int ph = rem / Wo, pw = rem - ph * Wo;
    const float* xp = x + static_cast<size_t>(n) * H * W;
    float in[4][4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int ih = 2 * ph + r - 1;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int iw = 2 * pw + c - 1;
        in[r][c] = (ih >= 0 && ih < H && iw >= 0 && iw < W) ? __ldg(xp + ih * W + iw) : 0.f;
      }
    }
    // packed fp32 FMAs on channel pairs (fma.rn.f32x2): the 16 inputs are duplicated into {x, x} once
    unsigned long long in2[4][4];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) asm("mov.b64 %0, {%1, %1};" : "=l"(in2[r][c]) : "f"(in[r][c]));
    uint4* op = reinterpret_cast<uint4*>(out + static_cast<size_t>(pix) * 64);
#pragma unroll
    for (int cg = 0; cg < 8; ++cg) {
      unsigned long long a[4][4];      // [pool position][channel pair]
#pragma unroll
      for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int j = 0; j < 4; ++j) a[q][j] = 0ull;
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        const int r = t / 3, s = t - 3 * (t / 3);
        const ulonglong2 w01 = *reinterpret_cast<const ulonglong2*>(&ws[t * 64 + cg * 8]);
        const ulonglong2 w23 = *reinterpret_cast<const ulonglong2*>(&ws[t * 64 + cg * 8 + 4]);
        const unsigned long long wv[4] = {w01.x, w01.y, w23.x, w23.y};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const unsigned long long v = in2[(q >> 1) + r][(q & 1) + s];
#pragma unroll
          for (int j = 0; j < 4; ++j) asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(a[q][j]) : "l"(v), "l"(wv[j]));
        }
      }
      float m[8];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float lo[4], hi[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) asm("mov.b64 {%0, %1}, %2;" : "=f"(lo[q]), "=f"(hi[q]) : "l"(a[q][j]));
        m[2 * j] = fmaxf(fmaxf(fmaxf(lo[0], lo[1]), fmaxf(lo[2], lo[3])) + bs[cg * 8 + 2 * j], 0.f);
        m[2 * j + 1] = fmaxf(fmaxf(fmaxf(hi[0], hi[1]), fmaxf(hi[2], hi[3])) + bs[cg * 8 + 2 * j + 1], 0.f);
      }
      op[cg] = make_uint4(pack_bf16x2(m[0], m[1]), pack_bf16x2(m[2], m[3]), pack_bf16x2(m[4], m[5]),
                          pack_bf16x2(m[6], m[7]));
    }
  }
}

// MaxPool2d(2,2) on bf16 NHWC: one thread = 8 channels of one output pixel (four 16 B loads, one
// 16 B store, coalesced along C).  HBM bound: 5/4 of the input bytes.
__global__ void __launch_bounds__(256) maxpool2x2_kernel(const __nv_bfloat16* __restrict__ in,
                                                         __nv_bfloat16* __restrict__ out, long long total_vec, int H,
                                                         int W, int C8) {
  const int Ho = H >> 1, Wo = W >> 1;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total_vec;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C8);
    long long t = i / C8;
    const int ow = static_cast<int>(t % Wo);
    t /= Wo;
    const int oh = static_cast<int>(t % Ho);
    const long long n = t / Ho;
    const uint4* p = reinterpret_cast<const uint4*>(in) + ((n * H + 2 * oh) * W + 2 * ow) * C8 + c;
    const uint4 v00 = __ldg(p), v01 = __ldg(p + C8), v10 = __ldg(p + static_cast<size_t>(W) * C8),
                v11 = __ldg(p + static_cast<size_t>(W) * C8 + C8);
    uint4 r;
    const uint32_t* a = &v00.x; const uint32_t* b = &v01.x; const uint32_t* c2 = &v10.x; const uint32_t* d = &v11.x;
    uint32_t* ro = &r.x;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const __nv_bfloat162 m0 = __hmax2(*reinterpret_cast<const __nv_bfloat162*>(a + j), *reinterpret_cast<const __nv_bfloat162*>(b + j));
      const __nv_bfloat162 m1 = __hmax2(*reinterpret_cast<const __nv_bfloat162*>(c2 + j), *reinterpret_cast<const __nv_bfloat162*>(d + j));
      const __nv_bfloat162 m = __hmax2(m0, m1);
      ro[j] = *reinterpret_cast<const uint32_t*>(&m);
    }
    reinterpret_cast<uint4*>(out)[i] = r;
  }
}

}  // namespace cer

using namespace cer;

struct cer_vggish {
  cer_vggish_weights w;
  std::vector<cer_vgg_conv> convs;
  std::vector<cer_vgg_fc> fcs;
  int64_t cap;
  int n_cap;
  int num_sms;
  uint8_t* buf[2];
  // kind 0: conv/fc, 1: pool (H, W, C: its input); desc: what cer_vggish_steps reports
  struct Step { int kind; ConvOp op; int H, W, C; const void* src; void* dst; cer_vggish_step desc; };
  std::vector<Step> steps;
  int emb_dim;
};

static const int kVggPad = 8;

// largest activation of the stack in bytes per patch (bf16)
static size_t vgg_max_act_bytes(const cer_vggish_weights* w) {
  int H = w->in_h / 2, W = w->in_w / 2;
  size_t mx = (size_t)H * W * w->c1 * 2;
  for (int i = 0; i < w->n_convs; ++i) {
    mx = std::max(mx, (size_t)H * W * w->convs[i].cout * 2);
    if (w->convs[i].pool_after) { H /= 2; W /= 2; }
  }
  for (int i = 0; i < w->n_fcs; ++i) mx = std::max(mx, (size_t)w->fcs[i].out_dim * 4);
  return mx;
}

extern "C" size_t cer_vggish_workspace_bytes(const cer_vggish_weights* w, int64_t patches_per_pass) {
  if (!w || patches_per_pass <= 0) return 0;
  const size_t act = ((vgg_max_act_bytes(w) * (patches_per_pass + kVggPad)) + 1023) & ~size_t(1023);
  return 2 * act + 1024;
}

extern "C" int cer_vggish_create(cer_vggish** out, const cer_vggish_weights* w, int64_t patches_per_pass,
                                 void* workspace_dev, size_t workspace_bytes) {
  if (!out || !w || !workspace_dev || patches_per_pass <= 0 || w->n_convs <= 0 || !w->convs || w->n_fcs <= 0 || !w->fcs ||
      !w->conv1_w || !w->conv1_bias || !w->zeros)
    return set_error(CER_ERR_INVALID, "cer_vggish_create: null/invalid argument");
  if (w->c1 != 64 || (w->in_h & 1) || (w->in_w & 1))
    return set_error(CER_ERR_INVALID, "cer_vggish_create: the first conv must have 64 outputs and even input sizes");
  if (patches_per_pass + kVggPad > (1 << 24)) return set_error(CER_ERR_INVALID, "patches_per_pass too large");
  int rc = cer_check_device();
  if (rc) return rc;
  rc = load_driver_entry_points();
  if (rc) return rc;
  if (workspace_bytes < cer_vggish_workspace_bytes(w, patches_per_pass))
    return set_error(CER_ERR_WORKSPACE, "cer_vggish_create: workspace too small");
  if (reinterpret_cast<uintptr_t>(workspace_dev) % 256) return set_error(CER_ERR_INVALID, "workspace must be 256B aligned");

  cer_vggish* p = new cer_vggish();
  p->w = *w;
  p->convs.assign(w->convs, w->convs + w->n_convs);
  p->fcs.assign(w->fcs, w->fcs + w->n_fcs);
  p->w.convs = p->convs.data();
  p->w.fcs = p->fcs.data();
  p->cap = patches_per_pass;
  p->n_cap = (int)patches_per_pass + kVggPad;
  int dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&p->num_sms, cudaDevAttrMultiProcessorCount, dev);
  const size_t act = ((vgg_max_act_bytes(w) * p->n_cap) + 1023) & ~size_t(1023);
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace_dev) + 1023) & ~uintptr_t(1023));
  p->buf[0] = base;
  p->buf[1] = base + act;

  int H = w->in_h / 2, W = w->in_w / 2, C = w->c1;
  int cur = 0;      // the stem writes buf[0]
  for (int i = 0; i < w->n_convs; ++i) {
    const cer_vgg_conv& c = p->convs[i];
    if (c.cin != C) { delete p; return set_error(CER_ERR_INVALID, "vggish: conv cin does not match the previous cout"); }
    ConvGeom g{};
    g.src = p->buf[cur]; g.H = H; g.W = W; g.Cin = c.cin; g.ksize = 3; g.stride = 1; g.pad = 1;
    g.weight = c.w; g.bias = c.bias; g.bias_classes = 1; g.alpha = w->zeros;      // PReLU slope 0 == ReLU
    g.dst = p->buf[cur ^ 1]; g.Cout = c.cout; g.out_fp32 = 0;
    const bool fuse_pool = c.pool_after && conv_can_pool(H, W, c.cin, c.cout) && !getenv("CER_NO_POOL_FUSION");
    g.pool = fuse_pool ? 1 : 0;
    cer_vggish::Step s{};
    s.kind = 0;
    rc = build_conv_op(&s.op, g, p->n_cap);
    if (rc) { delete p; return rc; }
    s.desc = {0, i, fuse_pool ? H / 2 : H, fuse_pool ? W / 2 : W, c.cout, 0, fuse_pool ? 1 : 0};
    p->steps.push_back(s);
    cur ^= 1;
    C = c.cout;
    if (fuse_pool) {          // the conv already wrote the pooled tensor
      H /= 2; W /= 2;
    } else if (c.pool_after) {
      if ((H & 1) || (W & 1) || (C % 8)) { delete p; return set_error(CER_ERR_INVALID, "vggish: pool needs even H, W and C % 8 == 0"); }
      cer_vggish::Step ps{};
      ps.kind = 1; ps.H = H; ps.W = W; ps.C = C; ps.src = p->buf[cur]; ps.dst = p->buf[cur ^ 1];
      ps.desc = {1, i, H / 2, W / 2, C, 0, 0};
      p->steps.push_back(ps);
      cur ^= 1;
      H /= 2; W /= 2;
    }
  }
  int dim = H * W * C;
  for (int i = 0; i < w->n_fcs; ++i) {
    const cer_vgg_fc& f = p->fcs[i];
    const bool last = i == w->n_fcs - 1;
    if (f.in_dim != dim || f.in_dim % 64 || f.out_dim % 64) { delete p; return set_error(CER_ERR_INVALID, "vggish: fc dims mismatch / not multiples of 64"); }
    ConvGeom g{};
    g.src = p->buf[cur]; g.H = 1; g.W = 1; g.Cin = f.in_dim; g.ksize = 1; g.stride = 1; g.pad = 0;
    g.weight = f.w; g.bias = f.bias; g.bias_classes = 1; g.alpha = f.relu ? w->zeros : nullptr;
    g.dst = p->buf[cur ^ 1]; g.Cout = f.out_dim; g.out_fp32 = last ? 1 : 0;
    cer_vggish::Step s{};
    s.kind = 0;
    rc = build_conv_op(&s.op, g, p->n_cap);
    if (rc) { delete p; return rc; }
    s.desc = {2, i, 1, 1, f.out_dim, last ? 1 : 0, 0};
    p->steps.push_back(s);
    cur ^= 1;
    dim = f.out_dim;
  }
  p->emb_dim = dim;
  *out = p;
  return CER_OK;
}

// One pass of n <= cap patches: the stem, then steps 0 .. last_step.  The last FC writes straight into emb_out.
static int run_pass(cer_vggish* p, const float* x, int n, int last_step, float* emb_out, cudaStream_t st) {
  const int H = p->w.in_h, W = p->w.in_w;
  const long long pix = (long long)n * (H / 2) * (W / 2);
  const int blocks = (int)std::min<long long>((pix + 127) / 128, (long long)p->num_sms * 16);
  vgg_stem_pool_kernel<<<blocks, 128, 0, st>>>(x, p->w.conv1_w, p->w.conv1_bias, reinterpret_cast<__nv_bfloat16*>(p->buf[0]),
                                               n, H, W);
  CER_CUDA(cudaGetLastError());
  for (size_t i = 0; i < p->steps.size() && (int)i <= last_step; ++i) {
    const cer_vggish::Step& s = p->steps[i];
    if (s.kind == 0) {
      if (i + 1 == p->steps.size()) {       // the last FC writes straight into the caller's output
        ConvOp op = s.op;
        op.kp.out = emb_out;
        int rc = launch_conv(op, n, p->num_sms, st);
        if (rc) return rc;
      } else {
        int rc = launch_conv(s.op, n, p->num_sms, st);
        if (rc) return rc;
      }
    } else {
      const int C8 = s.C / 8;
      const long long total = (long long)n * (s.H / 2) * (s.W / 2) * C8;
      const int pb = (int)std::min<long long>((total + 255) / 256, (long long)p->num_sms * 32);
      maxpool2x2_kernel<<<pb, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(s.src), static_cast<__nv_bfloat16*>(s.dst),
                                            total, s.H, s.W, C8);
      CER_CUDA(cudaGetLastError());
    }
  }
  return CER_OK;
}

extern "C" int cer_vggish_forward(cer_vggish* p, const float* x, int64_t n_patches, float* emb_out, void* stream) {
  if (!p || n_patches < 0 || (n_patches > 0 && (!x || !emb_out)))
    return set_error(CER_ERR_INVALID, "cer_vggish_forward: bad argument");
  // the last FC's epilogue stores 32-byte vectors straight into emb_out
  if (reinterpret_cast<uintptr_t>(x) % 4 || reinterpret_cast<uintptr_t>(emb_out) % 32)
    return set_error(CER_ERR_INVALID, "cer_vggish_forward: emb_out must be 32B aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int H = p->w.in_h, W = p->w.in_w;
  for (int64_t f0 = 0; f0 < n_patches; f0 += p->cap) {
    const int n = (int)std::min<int64_t>(p->cap, n_patches - f0);
    int rc = run_pass(p, x + f0 * H * W, n, (int)p->steps.size() - 1, emb_out + f0 * p->emb_dim, st);
    if (rc) return rc;
  }
  return CER_OK;
}

extern "C" int32_t cer_vggish_steps(const cer_vggish* p, cer_vggish_step* out, int32_t max_steps) {
  if (!p || max_steps < 0 || (max_steps > 0 && !out)) return set_error(CER_ERR_INVALID, "cer_vggish_steps: bad argument");
  for (int i = 0; i < (int)p->steps.size() && i < max_steps; ++i) out[i] = p->steps[i].desc;
  return (int32_t)p->steps.size();
}

extern "C" int64_t cer_vggish_debug_activation(cer_vggish* p, const float* x, int64_t n_patches, int32_t step, void* dst_dev,
                                               void* stream) {
  if (!p || !x || !dst_dev || n_patches <= 0 || n_patches > p->cap || step < -1 || step >= (int)p->steps.size())
    return set_error(CER_ERR_INVALID, "cer_vggish_debug_activation: bad argument");
  if (reinterpret_cast<uintptr_t>(x) % 4 || reinterpret_cast<uintptr_t>(dst_dev) % 32)   // the last FC stores into it
    return set_error(CER_ERR_INVALID, "cer_vggish_debug_activation: dst must be 32B aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool last = step + 1 == (int)p->steps.size();
  int rc = run_pass(p, x, (int)n_patches, step, last ? static_cast<float*>(dst_dev) : nullptr, st);
  if (rc) return rc;
  if (last) return n_patches * p->emb_dim;
  int64_t elems = n_patches * (p->w.in_h / 2) * (p->w.in_w / 2) * p->w.c1;
  const void* src = p->buf[0];
  if (step >= 0) {
    const cer_vggish::Step& s = p->steps[step];
    elems = n_patches * s.desc.h * s.desc.w * s.desc.c;
    src = s.kind == 0 ? s.op.kp.out : s.dst;
  }
  CER_CUDA(cudaMemcpyAsync(dst_dev, src, (size_t)elems * 2, cudaMemcpyDeviceToDevice, st));
  return elems;
}

extern "C" int cer_vggish_op_variant(const cer_vggish* p, int32_t step, int64_t n_patches, char* buf, int32_t buflen) {
  if (!p || !buf || buflen <= 0 || step < -1 || step >= (int)p->steps.size() || n_patches <= 0)
    return set_error(CER_ERR_INVALID, "cer_vggish_op_variant: bad argument");
  const int n = (int)std::min<int64_t>(p->cap, n_patches);
  const char* name = step < 0 ? "vgg_stem_pool_kernel"
                     : p->steps[step].kind == 1 ? "maxpool2x2_kernel"
                                                : conv_variant_name(p->steps[step].op, n, p->num_sms);
  const int len = snprintf(buf, (size_t)buflen, "%s", name);
  return len < buflen ? len : buflen - 1;
}

extern "C" int64_t cer_vggish_launches(const cer_vggish* p, int64_t n_patches) {
  if (!p || n_patches <= 0) return 0;
  const int64_t passes = (n_patches + p->cap - 1) / p->cap;
  return passes * (1 + (int64_t)p->steps.size());
}

extern "C" void cer_vggish_destroy(cer_vggish* p) { delete p; }
