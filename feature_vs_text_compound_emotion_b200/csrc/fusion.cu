// Fused cross-modal attention + LayerNorm + classifier, and the window-stitching kernel.
//
// Reference: MultimodalMultiheadAttention.forward (models/transformer.py:133-165),
// scaled_dot_product (:11-19), MultiModalEncoderBlock.forward (:192-197), then
// cat(leader, fused) -> regressor of LFAN.forward (models/model.py:517-521);
// window stitching: Trainer.inference_forward_windows (trainer.py:864-890).
//
// Per frame the "sequence" is the M modality tokens (M <= 4), head_dim 16: the whole op is a few
// tiny GEMVs.  One warp owns kFR frames at a time so each weight value read from shared memory is
// used kFR times; all weights (~150 KB fp32) are staged in shared memory once per CTA and the CTA
// grid-strides over frame groups.  Reductions (softmax over M, LayerNorm over E) use registers and
// warp shuffles only.  Memory-bound by design: compulsory traffic is (sum_m D_m + n_out) * 4 B per
// frame plus the weights once.
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdint>
#include <cmath>

#include "../../include/cer_b200.h"
#include "common.h"

namespace cer {

constexpr int kFRMin = 4, kFRMax = 8;   // frames per warp pass (template parameter kFR of the kernel, picked at launch)
constexpr int kFusWarps = 4;
constexpr int kFusThreads = kFusWarps * 32;
constexpr int kMaxE = 128;      // modal_dim * n_modals
constexpr int kMaxOut = 16;

// The instantiations cer_fusion_head_forward can run, kFR = 4..8 (cer_head_last_variant reports the one a launch used).
static const char* const kHeadVariantNames[] = {"fusion_head_kernel<4>", "fusion_head_kernel<5>", "fusion_head_kernel<6>",
                                                "fusion_head_kernel<7>", "fusion_head_kernel<8>"};

struct FusionDims {
  int M, E, D3, hd, H, n_out, din_total, dim[CER_MAX_MODALS], doff[CER_MAX_MODALS];
};

template <int kFR>
__global__ void __launch_bounds__(kFusThreads) fusion_head_kernel(cer_fusion_weights w, FusionDims d,
                                                                  const float* f0, const float* f1, const float* f2,
                                                                  const float* f3, long long rows,
                                                                  float* __restrict__ logits,
                                                                  float* __restrict__ fused_out) {
  extern __shared__ __align__(16) float sm[];
  // weights: wqkv (concatenated over modalities) | wo | wr | bqkv | bo | ln_g | ln_b | br
  float* s_wqkv = sm;                                 // [din_total][D3]
  float* s_wo = s_wqkv + d.din_total * d.D3;          // [E][E]
  float* s_wr = s_wo + d.E * d.E;                     // [dim0+E][n_out]
  float* s_bqkv = s_wr + (d.dim[0] + d.E) * d.n_out;  // [M][D3]
  float* s_bo = s_bqkv + d.M * d.D3;
  float* s_g = s_bo + d.E;
  float* s_b = s_g + d.E;
  float* s_br = s_b + d.E;                            // [n_out] (padded to 16)
  float* s_stage = s_br + kMaxOut;
  // per-warp staging: in [kFR][din_total] | qkv [kFR][M*D3] | vals [kFR][E]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int per_warp = kFR * (d.din_total + d.M * d.D3 + d.E);
  float* s_in = s_stage + warp * per_warp;
  float* s_qkv = s_in + kFR * d.din_total;
  float* s_val = s_qkv + kFR * d.M * d.D3;

  const float* feats[CER_MAX_MODALS] = {f0, f1, f2, f3};
  // Weight staging: ~145 KB per CTA.  A thread loop of LDG -> STS kept ~one load in flight per thread and took
  // 130 of the kernel's 150 us (ncu: every top stall an STS waiting on its LDG, profiles/r01_full_fusion.txt);
  // the TMA unit streams the same bytes with a handful of bulk copies onto one mbarrier (the host verified
  // 16-byte alignment and sizes: D3 and E*E are multiples of 4 floats).
  __shared__ __align__(8) unsigned long long s_bar;
  const uint32_t bar = static_cast<uint32_t>(__cvta_generic_to_shared(&s_bar));
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t total = static_cast<uint32_t>(d.E * d.E * 4);
    for (int m = 0; m < d.M; ++m) total += static_cast<uint32_t>(d.dim[m] * d.D3 * 4);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(total) : "memory");
    for (int m = 0; m <= d.M; ++m) {
      const float* src = m < d.M ? w.wqkv[m] : w.wo;
      float* dst = m < d.M ? s_wqkv + d.doff[m] * d.D3 : s_wo;
      uint32_t left = static_cast<uint32_t>((m < d.M ? d.dim[m] * d.D3 : d.E * d.E) * 4);
      uint32_t off = 0;
      while (left > 0) {                                    // pieces of at most 64 KB
        const uint32_t n = left < 65536u ? left : 65536u;
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(static_cast<uint32_t>(__cvta_generic_to_shared(reinterpret_cast<char*>(dst) + off))),
                       "l"(reinterpret_cast<const char*>(src) + off), "r"(n), "r"(bar)
                     : "memory");
        off += n; left -= n;
      }
    }
  }
  for (int i = threadIdx.x; i < (d.dim[0] + d.E) * d.n_out; i += kFusThreads) s_wr[i] = w.wr[i];
  for (int m = 0; m < d.M; ++m)
    for (int i = threadIdx.x; i < d.D3; i += kFusThreads) s_bqkv[m * d.D3 + i] = w.bqkv[m][i];
  for (int i = threadIdx.x; i < d.E; i += kFusThreads) { s_bo[i] = w.bo[i]; s_g[i] = w.ln_g[i]; s_b[i] = w.ln_b[i]; }
  if (threadIdx.x < d.n_out) s_br[threadIdx.x] = w.br[threadIdx.x];
  {
    uint32_t ok = 0;
    while (!ok) {
      asm volatile("{\n\t.reg .pred P;\n\tmbarrier.try_wait.parity.shared::cta.b64 P, [%1], 0;\n\tselp.b32 %0, 1, 0, P;\n\t}\n"
                   : "=r"(ok) : "r"(bar) : "memory");
    }
  }
  __syncthreads();

  const float scale = rsqrtf((float)d.hd);
  const long long groups = (rows + kFR - 1) / kFR;
  for (long long g = (long long)blockIdx.x * kFusWarps + warp; g < groups; g += (long long)gridDim.x * kFusWarps) {
    const long long r0 = g * kFR;
    // ---- stage inputs (zero for rows past the end)
    for (int m = 0; m < d.M; ++m) {
      const int dm = d.dim[m];
      for (int i = lane; i < kFR * dm; i += 32) {
        const int fr = i / dm, c = i - fr * dm;
        const long long r = r0 + fr;
        s_in[fr * d.din_total + d.doff[m] + c] = r < rows ? __ldg(feats[m] + r * dm + c) : 0.f;
      }
    }
    __syncwarp();
    // ---- qkv_m = b + f_m W_m      (lane owns output columns lane, lane+32, ...)
    for (int m = 0; m < d.M; ++m) {
      const float* wm = s_wqkv + d.doff[m] * d.D3;
      for (int j0 = 0; j0 < d.D3; j0 += 96) {        // up to 3 columns per lane per sweep
        float acc[3][kFR];
        int col[3];
#pragma unroll
        for (int q = 0; q < 3; ++q) {
          col[q] = j0 + lane + 32 * q;
          const float bq = col[q] < d.D3 ? s_bqkv[m * d.D3 + col[q]] : 0.f;
#pragma unroll
          for (int fr = 0; fr < kFR; ++fr) acc[q][fr] = bq;
          if (col[q] >= d.D3) col[q] = d.D3 - 1;     // clamp reads, result discarded
        }
        for (int i = 0; i < d.dim[m]; ++i) {
          float a[kFR];
#pragma unroll
          for (int fr = 0; fr < kFR; ++fr) a[fr] = s_in[fr * d.din_total + d.doff[m] + i];
#pragma unroll
          for (int q = 0; q < 3; ++q) {
            const float wv = wm[i * d.D3 + col[q]];
#pragma unroll
            for (int fr = 0; fr < kFR; ++fr) acc[q][fr] = fmaf(a[fr], wv, acc[q][fr]);
          }
        }
#pragma unroll
        for (int q = 0; q < 3; ++q) {
          const int c = j0 + lane + 32 * q;
          if (c < d.D3) {
#pragma unroll
            for (int fr = 0; fr < kFR; ++fr) s_qkv[(fr * d.M + m) * d.D3 + c] = acc[q][fr];
          }
        }
      }
    }
    __syncwarp();
    // ---- attention over the M modality tokens.  Output element e = (h, mq, dd) -> h*M*hd + mq*hd + dd
    //      qkv layout inside one modality: head h at h*3*hd: [q | k | v]   (transformer.py:142-144)
    for (int e = lane; e < d.E; e += 32) {
      const int h = e / (d.M * d.hd);
      const int mq = (e - h * d.M * d.hd) / d.hd;
      const int dd = e - h * d.M * d.hd - mq * d.hd;
#pragma unroll
      for (int fr = 0; fr < kFR; ++fr) {
        const float* base = s_qkv + fr * d.M * d.D3;
        const float* q = base + mq * d.D3 + h * 3 * d.hd;
        float sc[CER_MAX_MODALS];
        float mx = -INFINITY;
        for (int mk = 0; mk < d.M; ++mk) {
          const float* k = base + mk * d.D3 + h * 3 * d.hd + d.hd;
          float s = 0.f;
          for (int t = 0; t < d.hd; ++t) s = fmaf(q[t], k[t], s);
          sc[mk] = s * scale;
          mx = fmaxf(mx, sc[mk]);
        }
        float den = 0.f;
        for (int mk = 0; mk < d.M; ++mk) { sc[mk] = expf(sc[mk] - mx); den += sc[mk]; }
        float o = 0.f;
        for (int mk = 0; mk < d.M; ++mk) o = fmaf(sc[mk] / den, base[mk * d.D3 + h * 3 * d.hd + 2 * d.hd + dd], o);
        o += base[mq * d.D3 + h * 3 * d.hd + 2 * d.hd + dd];     // "+ V" residual (transformer.py:157)
        s_val[fr * d.E + e] = o;
      }
    }
    __syncwarp();
    // ---- o_proj + LayerNorm (lane owns columns lane, lane+32, lane+64, lane+96)
    float o[4][kFR];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int c = lane + 32 * q;
      const float bq = c < d.E ? s_bo[c] : 0.f;
#pragma unroll
      for (int fr = 0; fr < kFR; ++fr) o[q][fr] = bq;
    }
    for (int i = 0; i < d.E; ++i) {
      float a[kFR];
#pragma unroll
      for (int fr = 0; fr < kFR; ++fr) a[fr] = s_val[fr * d.E + i];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int c = lane + 32 * q;
        if (c < d.E) {
          const float wv = s_wo[i * d.E + c];
#pragma unroll
          for (int fr = 0; fr < kFR; ++fr) o[q][fr] = fmaf(a[fr], wv, o[q][fr]);
        }
      }
    }
    __syncwarp();
#pragma unroll
    for (int fr = 0; fr < kFR; ++fr) {
      float s = 0.f;
#pragma unroll
      for (int q = 0; q < 4; ++q) if (lane + 32 * q < d.E) s += o[q][fr];
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
      const float mean = s / d.E;
      float v = 0.f;
#pragma unroll
      for (int q = 0; q < 4; ++q) if (lane + 32 * q < d.E) { const float t = o[q][fr] - mean; v = fmaf(t, t, v); }
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
      const float rstd = rsqrtf(v / d.E + 1e-5f);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int c = lane + 32 * q;
        if (c < d.E) {
          const float y = (o[q][fr] - mean) * rstd * s_g[c] + s_b[c];
          s_val[fr * d.E + c] = y;            // fused feature, re-using the staging row
          if (fused_out != nullptr && r0 + fr < rows) fused_out[(r0 + fr) * d.E + c] = y;
        }
      }
    }
    __syncwarp();
    // ---- classifier on cat(leader features, fused):  logits[j] = br[j] + sum_i cat[i] * wr[i][j]
    const int dcat = d.dim[0] + d.E;
#pragma unroll
    for (int fr = 0; fr < kFR; ++fr) {
      float part[kMaxOut];
#pragma unroll
      for (int j = 0; j < kMaxOut; ++j) part[j] = 0.f;
      for (int i = lane; i < dcat; i += 32) {
        const float a = i < d.dim[0] ? s_in[fr * d.din_total + i] : s_val[fr * d.E + (i - d.dim[0])];
#pragma unroll
        for (int j = 0; j < kMaxOut; ++j)
          if (j < d.n_out) part[j] = fmaf(a, s_wr[i * d.n_out + j], part[j]);
      }
#pragma unroll
      for (int j = 0; j < kMaxOut; ++j) {
        if (j < d.n_out) {
#pragma unroll
          for (int off = 16; off > 0; off >>= 1) part[j] += __shfl_xor_sync(0xffffffffu, part[j], off);
        }
      }
      if (r0 + fr < rows) {
#pragma unroll
        for (int j = 0; j < kMaxOut; ++j)
          if (j < d.n_out && lane == j) logits[(r0 + fr) * d.n_out + j] = part[j] + s_br[j];
      }
    }
    __syncwarp();
  }
}

// out[t][c] = mean over windows covering t of win_logits[w][t - start_w][c]
__global__ void stitch_kernel(const float* __restrict__ win, const int* __restrict__ start, int n_windows, int win_len,
                              int n_out, long long length, float* __restrict__ out) {
  const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (idx >= length * n_out) return;
  const long long t = idx / n_out;
  const int c = (int)(idx - t * n_out);
  float s = 0.f;
  int cnt = 0;
  for (int w = 0; w < n_windows; ++w) {
    const long long rel = t - start[w];
    if (rel >= 0 && rel < win_len) {
      s += win[((size_t)w * win_len + rel) * n_out + c];
      ++cnt;
    }
  }
  out[idx] = cnt > 0 ? s / cnt : 0.f;
}

// Video-level decision rules of metrics.py:88-145 (format_trg_pred_video) for one video, one CTA:
// out[0] = FRAMES_VOTE (majority of per-frame argmax; ties -> the class seen first, as
// Counter.most_common), out[1] = FRAMES_AVG_LOGITS, out[2] = FRAMES_AVG_PROBS (row softmax, :43-48).
constexpr int kVoteMaxCls = 16;
__global__ void __launch_bounds__(256) video_vote_kernel(const float* __restrict__ logits, long long T, int n_cls_all,
                                                         int n_cls, int* __restrict__ out) {
  __shared__ float s_sum[8][kVoteMaxCls + 1];
  __shared__ float s_prob[8][kVoteMaxCls + 1];
  __shared__ int s_cnt[8][kVoteMaxCls + 1];
  __shared__ long long s_first[8][kVoteMaxCls + 1];
  float sum[kVoteMaxCls], prob[kVoteMaxCls];
  int cnt[kVoteMaxCls];
  long long first[kVoteMaxCls];
#pragma unroll
  for (int c = 0; c < kVoteMaxCls; ++c) { sum[c] = 0.f; prob[c] = 0.f; cnt[c] = 0; first[c] = T; }
  for (long long t = threadIdx.x; t < T; t += blockDim.x) {
    const float* p = logits + t * n_cls_all;
    float mx = p[0];
    int arg = 0;
    for (int c = 1; c < n_cls; ++c) if (p[c] > mx) { mx = p[c]; arg = c; }      // first maximum, like np.argmax
    float den = 0.f;
    for (int c = 0; c < n_cls; ++c) den += expf(p[c] - mx);
    const float inv = 1.f / den;
#pragma unroll
    for (int c = 0; c < kVoteMaxCls; ++c) {
      if (c < n_cls) {
        sum[c] += p[c];
        prob[c] += expf(p[c] - mx) * inv;
        if (c == arg) { ++cnt[c]; if (t < first[c]) first[c] = t; }
      }
    }
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int c = 0; c < kVoteMaxCls; ++c) {
    if (c < n_cls) {
      float a = sum[c], b = prob[c];
      int n = cnt[c];
      long long f = first[c];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
        n += __shfl_xor_sync(0xffffffffu, n, o);
        const long long f2 = __shfl_xor_sync(0xffffffffu, f, o);
        f = f2 < f ? f2 : f;
      }
      if (lane == 0) { s_sum[warp][c] = a; s_prob[warp][c] = b; s_cnt[warp][c] = n; s_first[warp][c] = f; }
    }
  }
  __syncthreads();
  if (threadIdx.x < n_cls) {
    const int c = threadIdx.x;
    float a = 0.f, b = 0.f;
    int n = 0;
    long long f = T;
    for (int i = 0; i < 8; ++i) {
      a += s_sum[i][c]; b += s_prob[i][c]; n += s_cnt[i][c];
      f = s_first[i][c] < f ? s_first[i][c] : f;
    }
    s_sum[0][c] = a; s_prob[0][c] = b; s_cnt[0][c] = n; s_first[0][c] = f;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int vote = 0, al = 0, ap = 0;
    for (int c = 1; c < n_cls; ++c) {
      if (s_cnt[0][c] > s_cnt[0][vote] || (s_cnt[0][c] == s_cnt[0][vote] && s_first[0][c] < s_first[0][vote])) vote = c;
      if (s_sum[0][c] > s_sum[0][al]) al = c;
      if (s_prob[0][c] > s_prob[0][ap]) ap = c;
    }
    out[0] = vote; out[1] = al; out[2] = ap;
  }
}

}  // namespace cer

extern "C" int cer_fusion_head_forward(const cer_fusion_weights* w, const float* const* feats, int64_t rows,
                                       float* logits, float* fused_out, void* stream) {
  using namespace cer;
  if (!w || !feats || !logits || rows < 0) return set_error(CER_ERR_INVALID, "cer_fusion_head_forward: bad argument");
  if (rows == 0) return CER_OK;
  FusionDims d{};
  d.M = w->n_modals;
  if (d.M < 1 || d.M > CER_MAX_MODALS) return set_error(CER_ERR_INVALID, "fusion: n_modals out of range");
  if (w->num_heads < 1 || w->modal_dim % w->num_heads) return set_error(CER_ERR_INVALID, "fusion: modal_dim % num_heads != 0");
  d.H = w->num_heads;
  d.hd = w->modal_dim / w->num_heads;
  d.D3 = 3 * w->modal_dim;
  d.E = w->modal_dim * d.M;
  d.n_out = w->n_out;
  if (d.E > kMaxE || d.n_out < 1 || d.n_out > kMaxOut) return set_error(CER_ERR_INVALID, "fusion: E > 128 or n_out > 16");
  int off = 0;
  for (int m = 0; m < d.M; ++m) {
    if (w->dim[m] <= 0 || !w->wqkv[m] || !w->bqkv[m] || !feats[m]) return set_error(CER_ERR_INVALID, "fusion: null modality input/weight");
    d.dim[m] = w->dim[m];
    d.doff[m] = off;
    off += w->dim[m];
  }
  d.din_total = off;
  if (!w->wo || !w->bo || !w->ln_g || !w->ln_b || !w->wr || !w->br) return set_error(CER_ERR_INVALID, "fusion: null weight");
  if (d.D3 % 4 || (d.E * d.E) % 4 || (reinterpret_cast<uintptr_t>(w->wo) & 15))
    return set_error(CER_ERR_INVALID, "fusion: modal_dim must be a multiple of 4 and weights 16B aligned");
  for (int m = 0; m < d.M; ++m)
    if (reinterpret_cast<uintptr_t>(w->wqkv[m]) & 15) return set_error(CER_ERR_INVALID, "fusion: wqkv must be 16B aligned");
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  constexpr size_t kMaxDyn = 227 * 1024 - 64;                 // the kernel's static mbarrier shares the 227 KB
  const size_t fixed = (size_t)d.din_total * d.D3 + (size_t)d.E * d.E + (size_t)(d.dim[0] + d.E) * d.n_out +
                       (size_t)d.M * d.D3 + 3 * (size_t)d.E + kMaxOut;
  const size_t per_frame = (size_t)kFusWarps * (d.din_total + d.M * d.D3 + d.E);
  auto smem_for = [&](int fr) { return (fixed + per_frame * fr) * sizeof(float); };
  if (smem_for(kFRMin) > kMaxDyn) return set_error(CER_ERR_INVALID, "fusion: weights do not fit in shared memory");
  // Frames per warp pass: every weight is read from shared memory once per pass whatever the frame count, so a
  // pass costs about the same for 4 or 8 frames.  Pick the smallest count for which ONE pass of the grid's
  // warps covers all rows (2400 rows: 5 frames x 592 warps; with 4 frames eight warps ran a second pass and
  // the kernel took twice as long, profiles/r02_fusion.txt), as far as shared memory allows.
  int fr = kFRMin;
  while (fr < kFRMax && (rows + fr - 1) / fr > (long long)sms * kFusWarps && smem_for(fr + 1) <= kMaxDyn) ++fr;
  const size_t smem = smem_for(fr);
  const long long groups = (rows + fr - 1) / fr;
  const int grid = (int)std::min<long long>((groups + kFusWarps - 1) / kFusWarps, sms);
  const float* f[CER_MAX_MODALS] = {nullptr, nullptr, nullptr, nullptr};
  for (int m = 0; m < d.M; ++m) f[m] = feats[m];
  cudaStream_t st = static_cast<cudaStream_t>(stream);
#define CER_FUSION_LAUNCH(FR)                                                                                              \
  case FR: {                                                                                                               \
    static unsigned long long configured = 0;                                                                              \
    if (first_use_on_device(&configured))                                                                                  \
      CER_CUDA(cudaFuncSetAttribute(fusion_head_kernel<FR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxDyn));   \
    set_head_variant(kHeadVariantNames[FR - kFRMin]);                                                                      \
    fusion_head_kernel<FR><<<grid, kFusThreads, smem, st>>>(*w, d, f[0], f[1], f[2], f[3], (long long)rows, logits, fused_out); \
  } break;
  switch (fr) {
    CER_FUSION_LAUNCH(4) CER_FUSION_LAUNCH(5) CER_FUSION_LAUNCH(6) CER_FUSION_LAUNCH(7) CER_FUSION_LAUNCH(8)
    default: return set_error(CER_ERR_INVALID, "fusion: frames per pass out of range");
  }
#undef CER_FUSION_LAUNCH
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

extern "C" int cer_stitch_windows(const float* win_logits, const int32_t* win_start, int32_t n_windows, int32_t win_len,
                                  int32_t n_out, int64_t length, float* out, void* stream) {
  using namespace cer;
  if (!win_logits || !win_start || !out || n_windows <= 0 || win_len <= 0 || n_out <= 0 || length <= 0)
    return set_error(CER_ERR_INVALID, "cer_stitch_windows: bad argument");
  const long long total = length * n_out;
  stitch_kernel<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      win_logits, win_start, n_windows, win_len, n_out, length, out);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

extern "C" int cer_video_vote(const float* logits_dev, int64_t length, int32_t n_cls, int32_t ignore_last_class,
                              int32_t* out_dev, void* stream) {
  using namespace cer;
  const int used = n_cls - (ignore_last_class ? 1 : 0);
  if (!logits_dev || !out_dev || length <= 0 || used < 1 || used > kVoteMaxCls)
    return set_error(CER_ERR_INVALID, "cer_video_vote: bad argument (1..16 classes, length >= 1)");
  video_vote_kernel<<<1, 256, 0, static_cast<cudaStream_t>(stream)>>>(logits_dev, length, n_cls, used, out_dev);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}
