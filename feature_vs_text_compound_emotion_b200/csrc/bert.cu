// BERT text encoder (HF BertModel in eval mode) for the `bert` feature stream, and the per-frame expansion of its
// token rows.  Transcripts of one call are laid end to end ("segments"), never padded:
//   embeddings   bert_embed_kernel: LayerNorm(word[id] + type[0] + pos[p]), eps from the config
//   per layer    qkv   = h Wqkv^T + b                      bert_linear_kernel, epilogue bias
//                ctx   = attention inside each segment     sdpa_tc_kernel<64, kSeg, kHeads> (heads.cu), one launch
//                t     = ctx Wo^T + bo + h                 bert_linear_kernel, epilogue bias + residual
//                a     = LayerNorm(t)                      cer_add_layernorm
//                inter = gelu(a W1^T + b1)                 bert_linear_kernel, epilogue bias + erf-GELU
//                t     = inter W2^T + b2 + a               bert_linear_kernel, epilogue bias + residual
//                h     = LayerNorm(t)                      cer_add_layernorm
//   output       sum of the last four hidden states (the layer outputs; with fewer than four layers the embedding
//                output counts, as hidden_states[-4:] of HF does), accumulated in the caller's fp32 buffer.
// The linear kernel is tcgen05.mma kind::tf32 with fp32 operands from TMA and the fp32 accumulator in TMEM, the
// pipeline of tcn_tc.cu with a tiled (not im2col) A operand.  Why TF32 and not bf16: SURVEY.md H4, as in tcn_tc.cu.
// One CTA owns one 128 x BN output tile over the whole K axis (no split-K), so a token's row takes the same
// instructions whatever else shares the call: every kernel here is row-invariant.
#include <cuda_runtime.h>
#include <cuda.h>
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../include/cer_b200.h"
#include "common.h"
#include "ptx.cuh"

namespace cer {

int make_tiled2d_map_generic(CUtensorMap* map, CUtensorMapDataType dt, int elem_bytes, const void* base, int rows,
                             int cols, int box_rows, int box_cols);

enum BertEpi { kEpiBias = 0, kEpiBiasGelu = 1, kEpiBiasRes = 2 };

struct alignas(64) BertLinearParams {
  CUtensorMap tmap_a;     // X [rows][K] fp32, box 128 x 32
  CUtensorMap tmap_b;     // W [N][K] fp32 (nn.Linear layout), box BN x 32
  int M, N, ksteps, num_n_tiles, epi;
  const float* bias;      // [N]
  const float* res;       // [M][N] (kEpiBiasRes)
  float* out;             // [M][N]
};

constexpr int kBlThreads = 256;       // warps 0-3 epilogue, 4 MMA, 5 A producer, 6 B producer, 7 idle
constexpr int kBlM = 128;
constexpr int kBlK = 32;              // 32 fp32 = 128 B = one swizzle row; 4 MMAs of K = 8 per k-step
constexpr int kBlABytes = kBlM * 128;

template <int BN, int STAGES>
struct BertLinearSmem {
  static constexpr int kBBytes = BN * 128;
  static constexpr int kStageBytes = kBlABytes + kBBytes;
  static constexpr int kBarOffset = STAGES * kStageBytes;
  static constexpr int kTotal = kBarOffset + (2 * STAGES + 2) * 8 + 16 + 1024;
};

__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.f + erff(x * 0.7071067811865476f)); }

// out[m, n] = epi(sum_k X[m, k] W[n, k] + bias[n]);  grid = ceil(M / 128) * N / BN, n tiles fastest.
template <int BN, int STAGES>
__global__ void __launch_bounds__(kBlThreads, 1) bert_linear_kernel(const __grid_constant__ BertLinearParams p) {
  using L = BertLinearSmem<BN, STAGES>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::kBarOffset);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* done_bar = empty_bar + STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done_bar + 2);
  constexpr uint32_t kTmemCols = BN;

  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const int m_tile = blockIdx.x / p.num_n_tiles;
  const int n_tile = blockIdx.x - m_tile * p.num_n_tiles;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 2);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(&done_bar[0], 1);
    fence_barrier_init();
  }
  if (warp == 5 && lane == 0) tma_prefetch_desc(&p.tmap_a);
  if (warp == 6 && lane == 0) tma_prefetch_desc(&p.tmap_b);
  if (warp == 4) {
    tmem_alloc(tmem_slot, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 5 || warp == 6) {
    // ---------------- TMA producers: warp 5 = A (activations), warp 6 = B (weights) ----------------
    const bool is_a = warp == 5;
    int stage = 0;
    uint32_t phase = 0;
    for (int ks = 0; ks < p.ksteps; ++ks) {
      mbar_wait(&empty_bar[stage], phase ^ 1);
      uint8_t* sa = smem + stage * L::kStageBytes;
      if (elect_one()) {
        if (is_a) {
          mbar_expect_tx(&full_bar[stage], kBlABytes);
          tma_load_2d(&p.tmap_a, &full_bar[stage], sa, ks * kBlK, m_tile * kBlM);
        } else {
          mbar_expect_tx(&full_bar[stage], L::kBBytes);
          tma_load_2d(&p.tmap_b, &full_bar[stage], sa + kBlABytes, ks * kBlK, n_tile * BN);
        }
      }
      __syncwarp();
      if (++stage == STAGES) { stage = 0; phase ^= 1; }
    }
  } else if (warp == 4) {
    // ---------------- MMA issuer ----------------
    constexpr uint32_t idesc = umma_idesc(kBlM, BN, /*tf32*/ 2);
    const uint32_t smem_base = smem_u32(smem);
    int stage = 0;
    uint32_t phase = 0;
    for (int ks = 0; ks < p.ksteps; ++ks) {
      mbar_wait(&full_bar[stage], phase);
      tc_fence_after();
      const uint32_t a_addr = smem_base + stage * L::kStageBytes;
      const uint64_t adesc = umma_desc_sw128(a_addr);
      const uint64_t bdesc = umma_desc_sw128(a_addr + kBlABytes);
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_tf32(tmem_base, adesc + 2 * k, bdesc + 2 * k, idesc, (ks == 0 && k == 0) ? 0u : 1u);
        umma_commit(&empty_bar[stage]);
        if (ks == p.ksteps - 1) umma_commit(&done_bar[0]);
      }
      __syncwarp();
      if (++stage == STAGES) { stage = 0; phase ^= 1; }
    }
  } else if (warp < 4) {
    // ---------------- Epilogue: one row per thread ----------------
    const int row = warp * 32 + lane;
    const uint32_t lane_addr = (static_cast<uint32_t>(warp * 32) << 16);
    const int m = m_tile * kBlM + row;
    const bool valid = m < p.M;
    const int n0 = n_tile * BN;
    const size_t off = static_cast<size_t>(m) * p.N + n0;
    mbar_wait(&done_bar[0], 0);
    tc_fence_after();
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      uint32_t v[32];
      tmem_ld_32x32(tmem_base + lane_addr + c0, v);
      tmem_ld_wait();
      float f[32];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + c0) + j);
        f[4 * j + 0] = __uint_as_float(v[4 * j + 0]) + b.x;
        f[4 * j + 1] = __uint_as_float(v[4 * j + 1]) + b.y;
        f[4 * j + 2] = __uint_as_float(v[4 * j + 2]) + b.z;
        f[4 * j + 3] = __uint_as_float(v[4 * j + 3]) + b.w;
      }
      if (p.epi == kEpiBiasGelu) {
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = gelu_erf(f[j]);
      } else if (p.epi == kEpiBiasRes && valid) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 x = __ldg(reinterpret_cast<const float4*>(p.res + off + c0) + j);
          f[4 * j + 0] += x.x; f[4 * j + 1] += x.y; f[4 * j + 2] += x.z; f[4 * j + 3] += x.w;
        }
      }
      if (valid) {
        float4* op = reinterpret_cast<float4*>(p.out + off + c0);
#pragma unroll
        for (int j = 0; j < 8; ++j) op[j] = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// BN = 128 when N allows it (2 CTAs of 3 stages per SM), else 64 (4 stages).
template <int BN, int STAGES>
static int launch_bert_linear(const BertLinearParams& p, int m_tiles, cudaStream_t st) {
  using L = BertLinearSmem<BN, STAGES>;
  static unsigned long long configured = 0;
  if (first_use_on_device(&configured))
    CER_CUDA(cudaFuncSetAttribute(bert_linear_kernel<BN, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kTotal));
  bert_linear_kernel<BN, STAGES><<<m_tiles * p.num_n_tiles, kBlThreads, L::kTotal, st>>>(p);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

static int bert_linear_bn(int n) { return n % 128 == 0 ? 128 : 64; }

static int run_bert_linear(const CUtensorMap& a, const CUtensorMap& b, int M, int N, int K, int epi, const float* bias,
                           const float* res, float* out, cudaStream_t st) {
  if (M == 0) return CER_OK;
  BertLinearParams p;
  memset(&p, 0, sizeof p);
  p.tmap_a = a;
  p.tmap_b = b;
  const int bn = bert_linear_bn(N);
  p.M = M; p.N = N; p.ksteps = K / kBlK; p.num_n_tiles = N / bn; p.epi = epi;
  p.bias = bias; p.res = res; p.out = out;
  const int m_tiles = (M + kBlM - 1) / kBlM;
  return bn == 128 ? launch_bert_linear<128, 3>(p, m_tiles, st) : launch_bert_linear<64, 4>(p, m_tiles, st);
}

// ---------------------------------------------------------------------------------------------------------------
// Embeddings: one warp per token.  grid (ceil(max_len / 8), n_seg); the token at position p of segment s is row
// seg_off[s] + p.  x = (word[id] + type[0]) + pos[p] (BertEmbeddings' order), then LayerNorm with lane-strided sums
// and an xor butterfly.  Products and sums use explicit round-to-nearest intrinsics (no FMA contraction), so the
// result is a fixed sequence of fp32 operations that a torch restatement reproduces bit for bit.  An id outside
// [0, vocab) reads nothing and gives a NaN row.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum_xor(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__global__ void __launch_bounds__(256) bert_embed_kernel(const int64_t* __restrict__ ids, const int32_t* __restrict__ seg_off,
                                                         int hidden, int vocab, const float* __restrict__ word,
                                                         const float* __restrict__ pos, const float* __restrict__ type0,
                                                         const float* __restrict__ gamma, const float* __restrict__ beta,
                                                         float eps, float* __restrict__ out) {
  const int s = blockIdx.y;
  const int p = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  const int row0 = seg_off[s];
  if (p >= seg_off[s + 1] - row0) return;
  const long long row = (long long)row0 + p;
  const long long id = ids[row];
  float* op = out + row * hidden;
  if (id < 0 || id >= vocab) {
    for (int i = lane; i < hidden; i += 32) op[i] = __int_as_float(0x7fc00000);
    return;
  }
  const float* wr = word + id * hidden;
  const float* pr = pos + (long long)p * hidden;
  float sum = 0.f;
  for (int i = lane; i < hidden; i += 32) sum = __fadd_rn(sum, __fadd_rn(__fadd_rn(wr[i], type0[i]), pr[i]));
  const float mean = __fdiv_rn(warp_sum_xor(sum), (float)hidden);
  float ss = 0.f;
  for (int i = lane; i < hidden; i += 32) {
    const float d = __fsub_rn(__fadd_rn(__fadd_rn(wr[i], type0[i]), pr[i]), mean);
    ss = __fadd_rn(ss, __fmul_rn(d, d));
  }
  const float rstd = __fdiv_rn(1.f, __fsqrt_rn(__fadd_rn(__fdiv_rn(warp_sum_xor(ss), (float)hidden), eps)));
  for (int i = lane; i < hidden; i += 32) {
    const float d = __fsub_rn(__fadd_rn(__fadd_rn(wr[i], type0[i]), pr[i]), mean);
    op[i] = __fadd_rn(__fmul_rn(__fmul_rn(d, rstd), gamma[i]), beta[i]);
  }
}

// Frame rows: out[f, :] = (rows[tok[f], :] - mean) / std, or the plain copy without mean / std.  One thread per
// 4 features, grid-stride.
__global__ void __launch_bounds__(256) text_frames_kernel(const float* __restrict__ rows, int ldr, const int32_t* __restrict__ tok,
                                                          long long n_frames, int dim, const float* __restrict__ mean,
                                                          const float* __restrict__ stdv, float* __restrict__ out, int ldo) {
  const int q = dim / 4;
  const long long total = n_frames * q;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long f = i / q;
    const int c = (int)(i - f * q) * 4;
    float4 x = __ldg(reinterpret_cast<const float4*>(rows + (long long)tok[f] * ldr + c));
    if (mean != nullptr) {
      const float4 m = __ldg(reinterpret_cast<const float4*>(mean + c));
      const float4 s = __ldg(reinterpret_cast<const float4*>(stdv + c));
      x = make_float4(__fdiv_rn(__fsub_rn(x.x, m.x), s.x), __fdiv_rn(__fsub_rn(x.y, m.y), s.y),
                      __fdiv_rn(__fsub_rn(x.z, m.z), s.z), __fdiv_rn(__fsub_rn(x.w, m.w), s.w));
    }
    *reinterpret_cast<float4*>(out + f * ldo + c) = x;
  }
}

}  // namespace cer

using namespace cer;

struct cer_bert {
  cer_bert_weights w;
  std::vector<cer_bert_layer> layers;
  int64_t max_tokens;
  float *h, *qkv, *ctx, *t, *a, *inter;     // workspace: [max_tokens] x {H, 3H, H, H, H, I} (bert_ws_floats)
  CUtensorMap map_h, map_ctx, map_a, map_inter;
  std::vector<CUtensorMap> map_w;           // per layer: wqkv, wo, w1, w2
};

static int check_bert_weights(const cer_bert_weights* w) {
  if (!w || !w->layers || !w->word_emb || !w->pos_emb || !w->type_emb || !w->emb_ln_g || !w->emb_ln_b)
    return set_error(CER_ERR_INVALID, "cer_bert: null weight");
  if (w->hidden <= 0 || w->hidden % 64 || w->intermediate <= 0 || w->intermediate % 64 || w->n_heads <= 0 ||
      w->hidden != 64 * w->n_heads || w->n_layers <= 0 || w->vocab <= 0 || w->max_pos <= 0 || w->max_pos > 512 ||
      w->type_vocab <= 0)
    return set_error(CER_ERR_INVALID, "cer_bert: unsupported configuration (head_dim 64, hidden and intermediate "
                                      "multiples of 64, at most 512 positions)");
  for (int l = 0; l < w->n_layers; ++l) {
    const cer_bert_layer& L = w->layers[l];
    if (!L.wqkv || !L.bqkv || !L.wo || !L.bo || !L.ln1_g || !L.ln1_b || !L.w1 || !L.b1 || !L.w2 || !L.b2 || !L.ln2_g ||
        !L.ln2_b)
      return set_error(CER_ERR_INVALID, "cer_bert: null layer weight");
  }
  return CER_OK;
}

// Workspace floats per token: h, qkv, ctx, t, a, inter of struct cer_bert.
static size_t bert_ws_floats(const cer_bert_weights* w) { return 7 * (size_t)w->hidden + w->intermediate; }

extern "C" size_t cer_bert_workspace_bytes(const cer_bert_weights* w, int64_t max_tokens) {
  if (!w || max_tokens <= 0 || w->hidden <= 0 || w->intermediate <= 0) return 0;
  return (size_t)max_tokens * bert_ws_floats(w) * sizeof(float);
}

extern "C" int cer_bert_create(cer_bert** out, const cer_bert_weights* w, int64_t max_tokens, void* workspace_dev,
                               size_t workspace_bytes) {
  if (!out) return set_error(CER_ERR_INVALID, "cer_bert_create: null out");
  *out = nullptr;
  int rc = check_bert_weights(w);
  if (rc) return rc;
  if (max_tokens <= 0 || max_tokens > (1 << 24)) return set_error(CER_ERR_INVALID, "cer_bert_create: max_tokens out of range");
  if (!workspace_dev || workspace_bytes < cer_bert_workspace_bytes(w, max_tokens))
    return set_error(CER_ERR_WORKSPACE, "cer_bert_create: workspace too small");
  if (reinterpret_cast<uintptr_t>(workspace_dev) % 16) return set_error(CER_ERR_INVALID, "cer_bert_create: workspace must be 16B aligned");
  rc = cer_check_device();
  if (rc) return rc;
  cer_bert* b = new cer_bert();
  b->w = *w;
  b->layers.assign(w->layers, w->layers + w->n_layers);
  b->w.layers = b->layers.data();
  b->max_tokens = max_tokens;
  const int H = w->hidden, I = w->intermediate, M = (int)max_tokens;
  float* base = static_cast<float*>(workspace_dev);
  b->h = base;
  b->qkv = b->h + (size_t)M * H;
  b->ctx = b->qkv + (size_t)M * 3 * H;
  b->t = b->ctx + (size_t)M * H;
  b->a = b->t + (size_t)M * H;
  b->inter = b->a + (size_t)M * H;
  const CUtensorMapDataType F = CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  rc = make_tiled2d_map_generic(&b->map_h, F, 4, b->h, M, H, kBlM, kBlK);
  if (!rc) rc = make_tiled2d_map_generic(&b->map_ctx, F, 4, b->ctx, M, H, kBlM, kBlK);
  if (!rc) rc = make_tiled2d_map_generic(&b->map_a, F, 4, b->a, M, H, kBlM, kBlK);
  if (!rc) rc = make_tiled2d_map_generic(&b->map_inter, F, 4, b->inter, M, I, kBlM, kBlK);
  b->map_w.resize(4 * (size_t)w->n_layers);
  for (int l = 0; l < w->n_layers && !rc; ++l) {
    const cer_bert_layer& L = b->layers[l];
    CUtensorMap* m = &b->map_w[4 * (size_t)l];
    rc = make_tiled2d_map_generic(m + 0, F, 4, L.wqkv, 3 * H, H, bert_linear_bn(3 * H), kBlK);
    if (!rc) rc = make_tiled2d_map_generic(m + 1, F, 4, L.wo, H, H, bert_linear_bn(H), kBlK);
    if (!rc) rc = make_tiled2d_map_generic(m + 2, F, 4, L.w1, I, H, bert_linear_bn(I), kBlK);
    if (!rc) rc = make_tiled2d_map_generic(m + 3, F, 4, L.w2, H, I, bert_linear_bn(H), kBlK);
  }
  if (rc) {
    delete b;
    return rc;
  }
  *out = b;
  return CER_OK;
}

extern "C" int cer_bert_forward(cer_bert* b, const int64_t* ids_dev, const int32_t* seg_off_dev, int32_t n_seg, int32_t max_len,
                                int64_t n_tokens, float* out_dev, void* stream) {
  if (!b || !ids_dev || !seg_off_dev || !out_dev || n_seg < 0 || max_len < 0 || n_tokens < 0)
    return set_error(CER_ERR_INVALID, "cer_bert_forward: bad argument");
  if (n_tokens > b->max_tokens) return set_error(CER_ERR_INVALID, "cer_bert_forward: more tokens than the plan's max_tokens");
  if (max_len > b->w.max_pos) return set_error(CER_ERR_INVALID, "cer_bert_forward: a segment longer than max_position_embeddings");
  if (n_seg > 65535) return set_error(CER_ERR_INVALID, "cer_bert_forward: more than 65535 segments");
  if (reinterpret_cast<uintptr_t>(out_dev) % 16) return set_error(CER_ERR_INVALID, "cer_bert_forward: out must be 16B aligned");
  if (n_tokens == 0 || n_seg == 0 || max_len == 0) return CER_OK;
  int rc = cer_check_device();
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const cer_bert_weights& w = b->w;
  const int H = w.hidden, I = w.intermediate, M = (int)n_tokens;
  const size_t row_bytes = (size_t)M * H * sizeof(float);

  dim3 eg((max_len + 7) / 8, n_seg);
  bert_embed_kernel<<<eg, 256, 0, st>>>(ids_dev, seg_off_dev, H, w.vocab, w.word_emb, w.pos_emb, w.type_emb, w.emb_ln_g,
                                        w.emb_ln_b, w.ln_eps, b->h);
  CER_CUDA(cudaGetLastError());
  // hidden_states[j], j = 0 (embeddings) .. n_layers; the last four are summed
  const int first_summed = w.n_layers - 3 > 0 ? w.n_layers - 3 : 0;
  auto accumulate = [&](int j) -> int {
    if (j < first_summed) return CER_OK;
    if (j == first_summed) {
      CER_CUDA(cudaMemcpyAsync(out_dev, b->h, row_bytes, cudaMemcpyDeviceToDevice, st));
      return CER_OK;
    }
    return cer_add_inplace(out_dev, b->h, (int64_t)M * H, st);
  };
  rc = accumulate(0);
  for (int l = 0; l < w.n_layers && !rc; ++l) {
    const cer_bert_layer& L = b->layers[l];
    const CUtensorMap* mw = &b->map_w[4 * (size_t)l];
    rc = run_bert_linear(b->map_h, mw[0], M, 3 * H, H, kEpiBias, L.bqkv, nullptr, b->qkv, st);
    if (!rc) rc = cer_sdpa_tc_seg_heads_forward(b->qkv, 3 * H, b->qkv + H, 3 * H, b->qkv + 2 * H, 3 * H, seg_off_dev, n_seg,
                                                max_len, 64, w.n_heads, b->ctx, H, st);
    if (!rc) rc = run_bert_linear(b->map_ctx, mw[1], M, H, H, kEpiBiasRes, L.bo, b->h, b->t, st);
    if (!rc) rc = cer_add_layernorm(b->t, nullptr, M, H, L.ln1_g, L.ln1_b, w.ln_eps, b->a, st);
    if (!rc) rc = run_bert_linear(b->map_a, mw[2], M, I, H, kEpiBiasGelu, L.b1, nullptr, b->inter, st);
    if (!rc) rc = run_bert_linear(b->map_inter, mw[3], M, H, I, kEpiBiasRes, L.b2, b->a, b->t, st);
    if (!rc) rc = cer_add_layernorm(b->t, nullptr, M, H, L.ln2_g, L.ln2_b, w.ln_eps, b->h, st);
    if (!rc) rc = accumulate(l + 1);
  }
  return rc;
}

extern "C" void cer_bert_destroy(cer_bert* b) { delete b; }

extern "C" int cer_bert_embed(const cer_bert* b, const int64_t* ids_dev, const int32_t* seg_off_dev, int32_t n_seg,
                              int32_t max_len, float* out_dev, void* stream) {
  if (!b || !ids_dev || !seg_off_dev || !out_dev || n_seg < 0 || max_len < 0 || n_seg > 65535 || max_len > b->w.max_pos)
    return set_error(CER_ERR_INVALID, "cer_bert_embed: bad argument");
  if (n_seg == 0 || max_len == 0) return CER_OK;
  const cer_bert_weights& w = b->w;
  dim3 eg((max_len + 7) / 8, n_seg);
  bert_embed_kernel<<<eg, 256, 0, static_cast<cudaStream_t>(stream)>>>(ids_dev, seg_off_dev, w.hidden, w.vocab, w.word_emb,
                                                                       w.pos_emb, w.type_emb, w.emb_ln_g, w.emb_ln_b, w.ln_eps,
                                                                       out_dev);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

extern "C" int cer_bert_linear(const float* x_dev, int64_t rows, int32_t in_dim, const float* w_dev, const float* bias_dev,
                               int32_t out_dim, int32_t epi, const float* res_dev, float* y_dev, void* stream) {
  if (!x_dev || !w_dev || !bias_dev || !y_dev || rows < 0 || rows > (1 << 24) || in_dim <= 0 || in_dim % 64 ||
      out_dim <= 0 || out_dim % 64 || epi < 0 || epi > 2 || (epi == kEpiBiasRes && !res_dev))
    return set_error(CER_ERR_INVALID, "cer_bert_linear: bad argument (in_dim and out_dim multiples of 64, epi 0..2, "
                                      "epi 2 needs res)");
  if ((reinterpret_cast<uintptr_t>(x_dev) | reinterpret_cast<uintptr_t>(w_dev) | reinterpret_cast<uintptr_t>(bias_dev) |
       reinterpret_cast<uintptr_t>(res_dev) | reinterpret_cast<uintptr_t>(y_dev)) % 16)
    return set_error(CER_ERR_INVALID, "cer_bert_linear: pointers must be 16B aligned");
  if (rows == 0) return CER_OK;
  int rc = cer_check_device();
  if (rc) return rc;
  CUtensorMap a, wm;
  rc = make_tiled2d_map_generic(&a, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, x_dev, (int)rows, in_dim, kBlM, kBlK);
  if (!rc) rc = make_tiled2d_map_generic(&wm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, w_dev, out_dim, in_dim, bert_linear_bn(out_dim), kBlK);
  if (rc) return rc;
  return run_bert_linear(a, wm, (int)rows, out_dim, in_dim, epi, bias_dev, res_dev, y_dev, static_cast<cudaStream_t>(stream));
}

extern "C" int cer_text_frames(const float* rows_dev, int32_t ldr, const int32_t* tok_dev, int64_t n_frames, int32_t dim,
                               const float* mean_dev, const float* std_dev, float* out_dev, int32_t ldo, void* stream) {
  if (!rows_dev || !tok_dev || !out_dev || n_frames < 0 || dim <= 0 || dim % 4 || ldr < dim || ldo < dim || ldr % 4 ||
      ldo % 4 || (mean_dev == nullptr) != (std_dev == nullptr))
    return set_error(CER_ERR_INVALID, "cer_text_frames: bad argument (dim and pitches multiples of 4, mean and std "
                                      "both given or both null)");
  if ((reinterpret_cast<uintptr_t>(rows_dev) | reinterpret_cast<uintptr_t>(out_dev) | reinterpret_cast<uintptr_t>(mean_dev) |
       reinterpret_cast<uintptr_t>(std_dev)) % 16)
    return set_error(CER_ERR_INVALID, "cer_text_frames: pointers must be 16B aligned");
  if (n_frames == 0) return CER_OK;
  const long long total = n_frames * (dim / 4);
  const int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  text_frames_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(rows_dev, ldr, tok_dev, (long long)n_frames, dim,
                                                                            mean_dev, std_dev, out_dev, ldo);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}
