/* cer_b200.h -- C-ABI of libcer_b200.so: the B200 (sm_100a) LFAN inference hot path.
 *
 * The reference (sbelharbi/feature-vs-text-compound-emotion) has no FFI layer: its boundary for
 * this path is the torch.nn.Module surface (SURVEY.md section 8b).  The entry points below are
 * what the host-side mirrors of those modules bind (feature_vs_text_compound_emotion_b200/
 * modules.py via ctypes); each cites the reference code it replaces (paths relative to the
 * reference root).
 *
 * Conventions
 *   - every pointer named *_dev / inside a *_weights struct is a DEVICE pointer owned by the caller;
 *   - no entry point allocates device memory (workspaces are caller-provided, sized by the
 *     *_workspace_bytes functions), none synchronises the device; all work is enqueued on
 *     `stream` (a cudaStream_t passed as void*);
 *   - return value: 0 on success, a negative cer_status otherwise (cer_last_error() gives the text);
 *   - handles are not thread-safe; distinct handles may be used from distinct threads.
 *   - activations inside the library are NHWC bf16, accumulation fp32; the TCN/fusion head
 *     computes in fp32.
 */
#ifndef CER_B200_H_
#define CER_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum cer_status {
  CER_OK = 0,
  CER_ERR_INVALID = -1,   /* bad shape / null pointer / misaligned pointer            */
  CER_ERR_ARCH = -2,      /* device is not compute capability 10.x                     */
  CER_ERR_CUDA = -3,      /* a CUDA runtime/driver call failed                         */
  CER_ERR_WORKSPACE = -4  /* workspace too small                                       */
} cer_status;

const char* cer_last_error(void);
int cer_version(void);
/* 0 if the current device can run the kernels (sm_100), CER_ERR_ARCH otherwise. */
int cer_check_device(void);

/* ------------------------------------------------------------------------------------------
 * IR-50 frame encoder.   Replaces VisualBackbone.forward / Backbone.forward
 * (models/backbone.py:124-126, models/arcface_model.py:147-151) incl. bottleneck_IR
 * (arcface_model.py:44-60), the 5x5 output_layer (backbone.py:99-103) and l2_norm (:17-20).
 * Weights arrive pre-packed by feature_vs_text_compound_emotion_b200/packing.py:
 * ------------------------------------------------------------------------------------------ */
/* A MaxPool2d(1, s) shortcut with s = 2 (cin == depth: the first unit of IR-100 / IR-152) is passed as a
 * projection with identity columns: w2 = [w2 | I], bias2 unchanged, has_proj = 1.  Products by 1.0 are exact.
 * In an IR-SE unit (cer_ir_se) a stride-2 identity shortcut is passed as is (has_proj = 0): the SE tail reads
 * the strided input directly. */
typedef struct cer_ir_unit {
  int32_t cin, depth, stride;   /* bottleneck_IR(in_channel, depth, stride)                        */
  int32_t has_proj;             /* 1: 1x1/stride conv+BN shortcut fused as extra K columns of w2   */
  const void* w1;               /* bf16 [depth][9*cin]   res_layer.1 with res_layer.0 (BN) scale folded; K = (r,s,ci) */
  const float* bias1;           /* fp32 [9][depth]       BN shift pushed through conv1, per border class           */
  const float* alpha;           /* fp32 [depth]          res_layer.2 PReLU slopes                                   */
  const void* w2;               /* bf16 [depth][9*depth (+cin)]  res_layer.3 * BN scale (+ shortcut conv * its BN scale) */
  const float* bias2;           /* fp32 [depth]          res_layer.4 BN shift (+ shortcut BN shift)                 */
                                /* IR-SE unit with has_proj: fp32 [2][depth], res_layer.4 shift then shortcut shift */
} cer_ir_unit;

/* SEModule(depth, 16) of an IR-SE unit (bottleneck_IR_SE, models/arcface_model.py:23-41, 63-84): res_layer.5.
 * The unit computes r = BN(conv3x3(PReLU(conv3x3(BN(x))))), gate[n][c] = sigmoid(fc2 relu(fc1 mean_hw(r))) and
 * out = r * gate + shortcut(x).  A projection shortcut runs as its own 1x1 conv (the w2 columns after 9*depth). */
typedef struct cer_ir_se {
  int32_t hidden, reserved;     /* hidden = depth / 16 (<= 64); reserved = 0                        */
  const float* fc1;             /* fp32 [hidden][depth]  res_layer.5.fc1.weight                     */
  const float* fc2;             /* fp32 [depth][hidden]  res_layer.5.fc2.weight                     */
} cer_ir_se;

typedef struct cer_ir50_weights {
  int32_t in_h, in_w;           /* 40, 40                                                          */
  const float* stem_w;          /* fp32 [27][64]  input_layer.0 * input_layer.1 scale; row = (r*3+s)*3+ci */
  const float* stem_bias;       /* fp32 [64]                                                       */
  const float* stem_alpha;      /* fp32 [64]      input_layer.2                                    */
  int32_t n_units;
  const cer_ir_unit* units;     /* HOST array of n_units entries (device pointers inside)          */
  int32_t fc_in;                /* H*W*C of the last unit's output (5*5*512)                       */
  int32_t emb_dim;              /* 512                                                             */
  const void* fc_w;             /* bf16 [emb_dim][fc_in], K in NHWC (h,w,c) order; output_layer.{0,3,4} folded */
  const float* fc_bias;         /* fp32 [emb_dim]                                                  */
} cer_ir50_weights;

typedef struct cer_ir50 cer_ir50;

/* Bytes of device workspace for a plan that processes up to `frames_per_pass` frames per pass. */
size_t cer_ir50_workspace_bytes(const cer_ir50_weights* w, int64_t frames_per_pass);
/* Builds TMA descriptors and launch configs over `workspace_dev`.  The weight pointers and the
 * workspace must stay valid and unmoved for the life of the plan. */
int cer_ir50_create(cer_ir50** out, const cer_ir50_weights* w, int64_t frames_per_pass, void* workspace_dev,
                    size_t workspace_bytes);
/* The same for an IR-SE backbone: `se` is a HOST array of n_units entries (device pointers inside); NULL gives
 * exactly the plan of cer_ir50_workspace_bytes / cer_ir50_create.  The SE plan adds a [frames_per_pass][512] fp32
 * gate buffer to the workspace and does not run the padded-raster stage. */
size_t cer_ir50_workspace_bytes_se(const cer_ir50_weights* w, const cer_ir_se* se, int64_t frames_per_pass);
int cer_ir50_create_se(cer_ir50** out, const cer_ir50_weights* w, const cer_ir_se* se, int64_t frames_per_pass,
                       void* workspace_dev, size_t workspace_bytes);
/* x_nchw_dev: fp32 [n_frames][3][in_h][in_w] in [-1,1]; emb_out_dev: fp32 [n_frames][emb_dim],
 * unit L2 norm per row.  Any n_frames >= 0 (processed in passes). */
int cer_ir50_forward(cer_ir50* plan, const float* x_nchw_dev, int64_t n_frames, float* emb_out_dev, void* stream);
/* Debug/inspection: run the stem and units 0..unit_index (-1 = stem only) on `frames`
 * (<= frames_per_pass) frames and copy that unit's bf16 NHWC output to dst_dev
 * (frames*H*W*C bf16; always dense NHWC -- a unit the plan keeps as a padded raster in this pass,
 * see DESIGN.md section 5.13, is un-padded on the way).  Returns the element count or a negative cer_status. */
int64_t cer_ir50_debug_activation(cer_ir50* plan, const float* x_nchw_dev, int64_t frames, int32_t unit_index,
                                  void* dst_dev, void* stream);
/* Name of the kernel instantiation the plan launches for conv op `op_index` (0 .. 2*n_units - 1: conv1,
 * conv2 of each unit in order; 2*n_units: the FC; after it, in an SE plan, the projection convs of the IR-SE
 * transition units in unit order) when a pass holds min(n_frames, frames_per_pass) frames,
 * e.g. "conv_igemm2_kernel<256,6>".  Writes a NUL-terminated string, returns its length or a negative status. */
int cer_ir50_op_variant(const cer_ir50* plan, int32_t op_index, int64_t n_frames, char* buf, int32_t buflen);
/* Profiling aid: launch ops [first_op, last_op] of one pass in plan order (0 = stem, 1 .. 2*n_units = unit
 * convs, 2*n_units + 1 = FC) on `frames` <= frames_per_pass frames.  The plan's activation buffers must hold
 * an earlier forward of the same frames.  x_nchw_dev is read by op 0 only.  The conv2 op of an IR-SE unit also
 * runs that unit's projection conv and SE tail, so the full range 0 .. 2*n_units + 1 is one forward pass. */
int cer_ir50_run_ops(cer_ir50* plan, const float* x_nchw_dev, int64_t frames, int32_t first_op, int32_t last_op, void* stream);
/* Number of kernel launches one forward of n_frames enqueues (for bench accounting; depends on the pass sizes:
 * a pass that runs the padded-raster stage adds one pad-zeroing launch; an IR-SE unit adds its squeeze and
 * scale kernels and, for a transition unit, its projection conv). */
int64_t cer_ir50_launches(const cer_ir50* plan, int64_t n_frames);
void cer_ir50_destroy(cer_ir50* plan);

/* One convolution through the same tcgen05 implicit-GEMM kernel (tests, per-layer roofline runs).
 * src: bf16 NHWC [n_alloc][h][w][cin] (n_alloc >= n_frames is the allocated / tensor-map extent);
 * weight: bf16 [cout][ksize*ksize*cin] with K = (r,s,ci); bias: fp32 [bias_classes][cout]
 * (bias_classes 9 = border-class table, stride-1 pad-1 3x3 only); alpha: PReLU slopes or NULL;
 * res: bf16 [M][cout] residual or NULL; dst: bf16 (or fp32 if out_fp32) [M][cout],
 * M = n_frames*hout*wout.  cin, cout multiples of 64. */
int cer_conv_forward(const void* src_nhwc_dev, int32_t n_frames, int32_t n_alloc, int32_t h, int32_t w, int32_t cin,
                     const void* weight_dev, int32_t cout, int32_t ksize, int32_t stride, int32_t pad,
                     const float* bias_dev, int32_t bias_classes, const float* alpha_dev, const void* res_dev,
                     void* dst_dev, int32_t out_fp32, void* stream);
/* Name of the kernel instantiation the last cer_conv_forward call on this thread launched. */
const char* cer_conv_last_variant(void);

/* ------------------------------------------------------------------------------------------
 * VGGish audio backbone (the inline `logmel` modality).   Replaces AudioBackbone.forward /
 * VGGish.forward / VGG.forward (models/backbone.py:29-40, :59-66, :133-145): six conv3x3+ReLU
 * with four 2x2 max-pools (make_layers, :43-53), NHWC flatten (:34-37), Linear-ReLU-Linear-ReLU-
 * Linear (:20-27).  Weights arrive pre-packed by packing.pack_vggish.
 * ------------------------------------------------------------------------------------------ */
typedef struct cer_vgg_conv {
  int32_t cin, cout, pool_after;  /* conv3x3 pad 1 + ReLU, then MaxPool2d(2,2) if pool_after        */
  const void* w;                  /* bf16 [cout][9*cin], K = (r,s,ci)                                */
  const float* bias;              /* fp32 [cout]                                                     */
} cer_vgg_conv;

typedef struct cer_vgg_fc {
  int32_t in_dim, out_dim, relu;
  const void* w;                  /* bf16 [out_dim][in_dim]; the first FC's K is the (h,w,c) flatten */
  const float* bias;              /* fp32 [out_dim]                                                  */
} cer_vgg_fc;

typedef struct cer_vggish_weights {
  int32_t in_h, in_w;             /* 96 frames x 64 mel bands                                        */
  int32_t c1;                     /* outputs of the first conv (64); it is always followed by a pool */
  const float* conv1_w;           /* fp32 [9][c1]  features.0.weight, row = r*3+s                    */
  const float* conv1_bias;        /* fp32 [c1]                                                       */
  int32_t n_convs;
  const cer_vgg_conv* convs;      /* HOST array: features.3 .. features.13                           */
  int32_t n_fcs;
  const cer_vgg_fc* fcs;          /* HOST array: embeddings.0/2/4                                    */
  const float* zeros;             /* fp32 [max(cout, out_dim)] zeros: ReLU = PReLU with slope 0      */
} cer_vggish_weights;

typedef struct cer_vggish cer_vggish;

size_t cer_vggish_workspace_bytes(const cer_vggish_weights* w, int64_t patches_per_pass);
int cer_vggish_create(cer_vggish** out, const cer_vggish_weights* w, int64_t patches_per_pass, void* workspace_dev,
                      size_t workspace_bytes);
/* x_dev: fp32 [n_patches][in_h][in_w] log-mel examples; emb_out_dev: fp32 [n_patches][128]. */
int cer_vggish_forward(cer_vggish* plan, const float* x_dev, int64_t n_patches, float* emb_out_dev, void* stream);
int64_t cer_vggish_launches(const cer_vggish* plan, int64_t n_patches);
void cer_vggish_destroy(cer_vggish* plan);

/* One step of the plan after the stem, in launch order (tests / inspection). */
typedef struct cer_vggish_step {
  int32_t kind;                   /* 0: convs[layer] (3x3 + ReLU), 1: the separate MaxPool2d(2,2) after convs[layer], 2: fcs[layer] */
  int32_t layer;
  int32_t h, w, c;                /* per-patch output: bf16 NHWC [h][w][c]; an FC is [1][1][out_dim]                    */
  int32_t out_fp32;               /* 1: fp32 output (the last FC)                                                       */
  int32_t pool_fused;             /* 1: a conv whose epilogue applies the following MaxPool2d(2,2) (h, w are pooled)   */
} cer_vggish_step;
/* Copies the first min(max_steps, n) step descriptors to `out` and returns n, the number of steps. */
int32_t cer_vggish_steps(const cer_vggish* plan, cer_vggish_step* out, int32_t max_steps);
/* Debug/inspection: one pass over `n_patches` (<= patches_per_pass) patches -- the stem, then steps 0 .. step --
 * and a copy of that step's output to dst_dev (16 B aligned).  step = -1 is the stem's pooled bf16
 * [n][in_h/2][in_w/2][c1]; the last step (the fp32 FC) writes dst_dev directly.  At n_patches = patches_per_pass
 * the launches are exactly those of that cer_vggish_forward pass.  Returns the element count or a negative status. */
int64_t cer_vggish_debug_activation(cer_vggish* plan, const float* x_dev, int64_t n_patches, int32_t step, void* dst_dev,
                                    void* stream);
/* Name of the kernel instantiation step `step` launches when a pass holds min(n_patches, patches_per_pass) patches:
 * "vgg_stem_pool_kernel" for step -1, "maxpool2x2_kernel" for a separate pool, else a conv variant such as
 * "conv_igemm2_kernel<256,6>".  Writes a NUL-terminated string, returns its length or a negative status. */
int cer_vggish_op_variant(const cer_vggish* plan, int32_t step, int64_t n_patches, char* buf, int32_t buflen);

/* ------------------------------------------------------------------------------------------
 * Log-mel front end of the inline-VGGish modality.   Replaces log_mel_spectrogram /
 * stft_magnitude / periodic_hann / spectrogram_to_mel_matrix (abaw5_pre_processing/base/vggish/
 * mel_features.py:92-236) and the example framing my_frame (:21-46; vggish_input.py:70-79).
 * fp64 arithmetic like the numpy reference, fp32 output.
 * wave_dev: fp32 mono samples at the VGGish rate (16 kHz); tables_dev: fp64
 *   [win] periodic Hann | [fft] cos(2 pi i/fft) | [fft] sin(2 pi i/fft) | [fft/2+1][n_mel] mel matrix
 *   (built on the host by packing.logmel_tables with the reference's formulas);
 * logmel_out_dev: fp32 [cer_logmel_num_frames(n_samples, win, hop)][n_mel] = log(mel + log_offset).
 * cer_frame_examples: out[e][t][:] = logmel[starts[e] + t][:], e < n_examples, t < frames_per_example.
 * ------------------------------------------------------------------------------------------ */
int64_t cer_logmel_num_frames(int64_t n_samples, int32_t win, int32_t hop);
int cer_logmel_forward(const float* wave_dev, int64_t n_samples, const double* tables_dev, int32_t win, int32_t hop,
                       int32_t fft, int32_t n_mel, double log_offset, float* logmel_out_dev, void* stream);
int cer_frame_examples(const float* logmel_dev, const int32_t* starts_dev, int32_t n_examples, int32_t frames_per_example,
                       int32_t n_mel, float* out_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * One TemporalBlock, fused.   Replaces TemporalBlock.forward
 * (models/temporal_convolutional_model.py:21-54): weight-normed dilated Conv1d + Chomp1d +
 * LeakyReLU, twice, plus identity / 1x1 residual and the final LeakyReLU.  Optionally applies a
 * trailing per-channel affine (the eval BatchNorm1d of models/model.py:475,515) to the output.
 * Layout: x [B][T][c_in] fp32 (time-major rows, channels contiguous), y [B][T][c_out] fp32.
 * ------------------------------------------------------------------------------------------ */
typedef struct cer_tcn_block {
  int32_t c_in, c_out, kernel_size, dilation;
  const float* w1;      /* fp32 [k][c_in][c_out]   effective (g*v/||v||) conv1 weight, tap-major        */
  const float* b1;      /* fp32 [c_out]                                                                  */
  const float* w2;      /* fp32 [k][c_out][c_out]  effective conv2 weight                                */
  const float* b2;      /* fp32 [c_out]                                                                  */
  const float* wd;      /* fp32 [c_in][c_out]      1x1 downsample or NULL (identity residual)            */
  const float* bd;      /* fp32 [c_out] or NULL                                                          */
  const float* post_scale; /* fp32 [c_out] or NULL: y = y*post_scale + post_shift after the last LeakyReLU */
  const float* post_shift;
} cer_tcn_block;

size_t cer_tcn_block_workspace_bytes(const cer_tcn_block* blk, int64_t batch, int64_t length);
int cer_tcn_block_forward(const cer_tcn_block* blk, const float* x_dev, float* y_dev, int64_t batch, int64_t length,
                          void* workspace_dev, size_t workspace_bytes, void* stream);

/* Tensor-core variant (tcgen05 kind::tf32: fp32 operands, 10-bit-mantissa multiply, fp32
 * accumulate) -- the production path.  Same struct, different weight layout:
 *   w1: fp32 [c_out][k*c_in], K = (tap, ci);   w2: fp32 [c_out][k*c_out (+ c_in)] with the 1x1
 *   downsample weights appended as the last c_in columns (wd != NULL only flags their presence,
 *   bd is its bias).  Channels must be multiples of 32, the causal halo (kernel_size-1)*dilation at most 128
 *   (the im2col tensor map's bounding-box corner range).  workspace holds conv1's output. */
size_t cer_tcn_block_tc_workspace_bytes(const cer_tcn_block* blk, int64_t batch, int64_t length);
int cer_tcn_block_tc_forward(const cer_tcn_block* blk, const float* x_dev, float* y_dev, int64_t batch, int64_t length,
                             void* workspace_dev, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Cross-modal attention fusion + classifier, fused.   Replaces
 * MultimodalTransformerEncoder.forward (models/transformer.py:200-209, :168-197, :102-165,
 * :11-19) followed by cat + regressor of LFAN.forward (models/model.py:517-521).
 * feats[m]: fp32 [rows][dim[m]] (rows = B*T frames); logits: fp32 [rows][n_out].
 * ------------------------------------------------------------------------------------------ */
#define CER_MAX_MODALS 4
typedef struct cer_fusion_weights {
  int32_t n_modals;                 /* 1..CER_MAX_MODALS; modality 0 is the leader              */
  int32_t dim[CER_MAX_MODALS];      /* encoder_dim per modality (128, 32, 128)                   */
  int32_t modal_dim, num_heads;     /* 32, 2                                                     */
  int32_t n_out;                    /* classifier outputs (7)                                    */
  const float* wqkv[CER_MAX_MODALS];/* fp32 [dim[m]][3*modal_dim]  qkv_proj.<m>.weight transposed */
  const float* bqkv[CER_MAX_MODALS];/* fp32 [3*modal_dim]                                         */
  const float* wo;                  /* fp32 [E][E] o_proj.weight transposed (in-major), E = modal_dim*n_modals */
  const float* bo;                  /* fp32 [E]                                                   */
  const float* ln_g;                /* fp32 [E] norm1.weight                                      */
  const float* ln_b;                /* fp32 [E] norm1.bias                                        */
  const float* wr;                  /* fp32 [dim[0]+E][n_out] regressor.weight transposed         */
  const float* br;                  /* fp32 [n_out]                                               */
} cer_fusion_weights;

/* Attention probabilities of the cross-modal attention (MultimodalTransformerEncoder.get_attention_maps,
 * transformer.py:211-215 -> scaled_dot_product :11-19).  qkv_dev[m]: fp32 [rows][3*modal_dim] = qkv_proj.<m>(x_m)
 * (cer_linear_forward), per head laid out q|k|v; maps_out_dev: fp32 [rows][num_heads][n_modals][n_modals]. */
int cer_modal_attention_maps(const float* const* qkv_dev, int64_t rows, int32_t n_modals, int32_t num_heads, int32_t head_dim,
                             float* maps_out_dev, void* stream);

/* The attention itself for configurations whose weights do not fit the fused kernel's shared memory:
 * vals_out_dev fp32 [rows][n_modals*num_heads*head_dim] = softmax(QK^T/sqrt(hd))V + V, packed (head, modal, dim)
 * (transformer.py:150-159); combine with cer_linear_forward (qkv_proj, o_proj, regressor) and cer_add_layernorm. */
int cer_modal_attention_forward(const float* const* qkv_dev, int64_t rows, int32_t n_modals, int32_t num_heads,
                                int32_t head_dim, float* vals_out_dev, void* stream);

int cer_fusion_head_forward(const cer_fusion_weights* w, const float* const* feats_dev, int64_t rows,
                            float* logits_dev, float* fused_out_dev /* [rows][E] or NULL */, void* stream);

/* Name of the kernel instantiation the last head launch on this thread ran: one conv launch of
 * cer_tcn_block_tc_forward (e.g. "tcn_igemm_kernel<64,8>"), cer_tcn_block_forward ("tcn_block_kernel<128,4,5>")
 * or cer_fusion_head_forward ("fusion_head_kernel<5>").  "none" before the first launch; a call refused
 * before launching leaves it unchanged. */
const char* cer_head_last_variant(void);

/* ------------------------------------------------------------------------------------------
 * Fusion-head training step (BASELINE config 4).   Replaces, for the trainable head of LFAN
 * (TCN x M, BatchNorm1d, cross-modal attention, LayerNorm, classifier), the forward in
 * training mode + loss + backward + optimizer step of trainer.py:365-391 / experiment.py:133 /
 * instantiators.py:60-100.  Exact fp32.  Parameters are read in the reference's own layouts
 * (weight_g [cout], weight_v [cout][cin][k], Linear weight [out][in]); gradients are written in
 * the same layouts.  All gradient pointers must lie inside one flat buffer [grad_flat,
 * grad_flat + grad_count) (zeroed by backward; one NCCL all-reduce covers it).
 * Dropout masks come from a counter hash of (seed, site, element) that oracle/lfan_oracle.py
 * restates; p_tcn = p_fusion = 0 disables dropout.
 * ------------------------------------------------------------------------------------------ */
#define CER_MAX_TCN_BLOCKS 6
typedef struct cer_train_conv {
  const float *g, *v, *bias;        /* weight_g [cout], weight_v [cout][cin][k], bias [cout]       */
  float *dg, *dv, *dbias;
} cer_train_conv;

typedef struct cer_train_block {
  int32_t c_in, c_out, dilation, reserved;
  cer_train_conv conv1, conv2;
  const float *wd, *bd;             /* downsample.weight [cout][cin] / bias, NULL when c_in == c_out */
  float *dwd, *dbd;
} cer_train_block;

typedef struct cer_train_modal {
  int32_t in_dim, n_blocks;
  cer_train_block blocks[CER_MAX_TCN_BLOCKS];
  const float *bn_w, *bn_b;         /* bn.<m>.weight / bias                                          */
  float *dbn_w, *dbn_b;
  float *bn_mean, *bn_var;          /* running statistics, updated in place by forward               */
  const float *wqkv, *bqkv;         /* qkv_proj.<m>.weight [3*modal_dim][c_last], bias               */
  float *dwqkv, *dbqkv;
} cer_train_modal;

typedef struct cer_head_train_spec {
  int32_t n_modals, kernel_size, modal_dim, num_heads, n_out;
  int32_t precision;            /* 0: exact fp32 GEMMs (CUDA cores); 1: the TCN convolutions (forward, dgrad, wgrad) on TF32
                                 * tensor cores with fp32 accumulate -- torch's own GPU default for convolutions; the fusion
                                 * head's Linear layers stay fp32 */
  double p_tcn, p_fusion, bn_momentum;   /* 0.1, 0.1, 0.1 in the reference (model.py:471,482)        */
  cer_train_modal modal[CER_MAX_MODALS]; /* modality 0 is the leader                                 */
  const float *wo, *bo, *ln_g, *ln_b, *wr, *br;
  float *dwo, *dbo, *dln_g, *dln_b, *dwr, *dbr;
  float* grad_flat;
  int64_t grad_count;
} cer_head_train_spec;

typedef struct cer_head_train cer_head_train;

size_t cer_head_train_workspace_bytes(const cer_head_train_spec* spec, int64_t batch, int64_t length);
int cer_head_train_create(cer_head_train** out, const cer_head_train_spec* spec, int64_t batch, int64_t length,
                          void* workspace_dev, size_t workspace_bytes);
/* feats_dev[m]: fp32 [batch*length][in_dim[m]] time-major rows; logits_dev: fp32 [batch*length][n_out].
 * Saves the activations backward needs in the workspace and updates the BatchNorm running stats. */
int cer_head_train_forward(cer_head_train* plan, const float* const* feats_dev, uint32_t seed, float* logits_dev, void* stream);
/* dlogits_dev: fp32 [batch*length][n_out] = d loss / d logits; writes every gradient of the spec. */
int cer_head_train_backward(cer_head_train* plan, const float* const* feats_dev, const float* dlogits_dev, void* stream);
void cer_head_train_destroy(cer_head_train* plan);
/* The TemporalConvNet + BatchNorm1d part of the plan alone -- what CAN / JMT / MT share with LFAN
 * (models/model.py:672-676, :1155-1159): z_dev[m] receives fp32 [batch*length][c_last[m]] (dense).  The fusion
 * fields of the spec (wo ... dbr, wqkv ...) may be NULL in a plan that is only used through these two calls. */
int cer_head_train_tcn_forward(cer_head_train* plan, const float* const* feats_dev, uint32_t seed, float* const* z_dev, void* stream);
/* dz_dev[m] = d loss / d z[m].  Unlike cer_head_train_backward this does NOT clear the flat gradient buffer: the caller
 * zeroes it once per step and the other blocks of the head add into it. */
int cer_head_train_tcn_backward(cer_head_train* plan, const float* const* feats_dev, const float* const* dz_dev, void* stream);

/* ---- building blocks WITH backward, for training CAN / JMT / MT (experiment.py:317-347 trains them through the same loop).
 * Parameter gradients are ACCUMULATED (+=) into caller-zeroed buffers; activation gradients are written. ---- */
/* y = x W^T + b: dx[rows][in] (= or += if dx_accumulate) = dy W; dw[out][in] += dy^T x; db[out] += column sums of dy.
 * Any of dx / dw / db may be NULL. */
int cer_linear_backward(const float* x_dev, int64_t rows, int32_t in_dim, int32_t ldx, const float* w_dev, const float* dy_dev,
                        int32_t out_dim, int32_t lddy, float* dx_dev, int32_t lddx, int32_t dx_accumulate, float* dw_dev, float* db_dev,
                        void* stream);
/* dx = dy * act'(.) from the saved OUTPUT y of the activation: act 1 = LeakyReLU(0.01), 2 = ReLU. */
int cer_act_backward(int32_t act, const float* y_dev, const float* dy_dev, int64_t n, float* dx_dev, void* stream);
int cer_leaky_relu_forward(const float* x_dev, int64_t n, float* y_dev, void* stream);
/* backward of cer_softmax_gate (AttentionFusion, model.py:563-567) */
int cer_softmax_gate_backward(const float* gate_dev, const float* feat_dev, const float* dy_dev, int64_t rows, int32_t dim,
                              float* dgate_dev, float* dfeat_dev, void* stream);
/* backward of cer_add_layernorm: dx (which is also d res), dgamma +=, dbeta +=; dim <= 512 */
int cer_add_layernorm_backward(const float* x_dev, const float* res_dev, int64_t rows, int32_t dim, const float* gamma_dev, float eps,
                               const float* dy_dev, float* dx_dev, float* dgamma_dev, float* dbeta_dev, void* stream);
/* nn.BatchNorm1d in training mode over [rows][c] (batch statistics, running-stat update with the unbiased variance) */
int cer_bn1d_train_forward(const float* x_dev, int64_t rows, int32_t c, const float* w_dev, const float* b_dev, float* y_dev,
                           float* save_mean_dev, float* save_invstd_dev, float* running_mean_dev, float* running_var_dev, float momentum,
                           void* stream);
int cer_bn1d_train_backward(const float* dy_dev, const float* x_dev, int64_t rows, int32_t c, const float* w_dev,
                            const float* save_mean_dev, const float* save_invstd_dev, float* dx_dev, float* dw_dev, float* db_dev,
                            void* stream);
/* single-head attention keeping the probabilities [batch][len_q][len_k] for backward (exact fp32 GEMMs) */
int cer_sdpa_train_forward(const float* q_dev, int32_t ldq, const float* k_dev, int32_t ldk, const float* v_dev, int32_t ldv,
                           int32_t batch, int32_t len_q, int32_t len_k, int32_t dim, float* out_dev, int32_t ldo, float* probs_dev,
                           void* stream);
/* dq is written, dk / dv are accumulated (zero them first); scratch_dev: [batch][len_q][len_k] floats */
int cer_sdpa_backward(const float* q_dev, int32_t ldq, const float* k_dev, int32_t ldk, const float* v_dev, int32_t ldv,
                      const float* probs_dev, const float* dout_dev, int32_t lddo, int32_t batch, int32_t len_q, int32_t len_k,
                      int32_t dim, float* dq_dev, int32_t lddq, float* dk_dev, int32_t lddk, float* dv_dev, int32_t lddv,
                      float* scratch_dev, void* stream);

/* Mean cross-entropy over `rows` rows (<= 2^20) and (optionally) its gradient w.r.t. the logits
 * (nn.CrossEntropyLoss(reduction="mean"), experiment.py:133).  labels: int64 [rows].  Rows whose label is
 * ignore_index (-100) are excluded from the mean and get a zero gradient, as in torch; any other label
 * outside [0, n_cls) is treated the same way (torch raises a device assert there) -- it is never used as
 * an index.  With no valid row the loss is NaN, as in torch. */
int cer_ce_loss(const float* logits_dev, const int64_t* labels_dev, int64_t rows, int32_t n_cls, float* loss_out_dev,
                float* dlogits_out_dev /* or NULL */, void* stream);

/* Fused optimizer update over a flat fp32 buffer.  kind 0: SGD (beta1 = momentum, beta2 = dampening,
 * nesterov), 1: Adam, 2: AdamW -- torch.optim arithmetic (instantiators.py:60-100).  step counts
 * from 1.  grads are multiplied by grad_scale first (1/world_size after a sum all-reduce). */
int cer_optimizer_step(int32_t kind, float* params_dev, const float* grads_dev, float* state_m_dev, float* state_v_dev,
                       int64_t n, float lr, float weight_decay, float beta1_or_momentum, float beta2_or_dampening, float eps,
                       int32_t nesterov, int32_t step, float grad_scale, void* stream);

/* ------------------------------------------------------------------------------------------
 * Eval-time input pipeline.   Replaces the video transform of base/dataset.py:503-510
 * (GroupNumpyToPILImage -> GroupScale(48) -> GroupCenterCrop(40) -> Stack -> ToTorchFormatTensor
 * -> GroupNormalize(.5,.5); base/transforms3D.py:15-144) including Pillow's antialiased 8-bit
 * BILINEAR resize, bit-exactly, for the crop window only.
 * frames_dev: uint8 [n][in_h][in_w][3] as stored (video.npy); out_dev: fp32 [n][3][crop][crop].
 * cer_preproc_create copies its coefficient tables into workspace_dev (cer_preproc_workspace_bytes
 * bytes, caller-owned, must outlive the plan) with a synchronous cudaMemcpy.
 * ------------------------------------------------------------------------------------------ */
typedef struct cer_preproc cer_preproc;
size_t cer_preproc_workspace_bytes(void);
int cer_preproc_create(cer_preproc** out, int32_t in_h, int32_t in_w, int32_t resize, int32_t crop, void* workspace_dev,
                       size_t workspace_bytes);
int cer_preproc_forward(cer_preproc* plan, const uint8_t* frames_dev, int64_t n_frames, float* out_dev, void* stream);
void cer_preproc_destroy(cer_preproc* plan);

/* ------------------------------------------------------------------------------------------
 * Building blocks of the alternative fusion heads CAN / JMT / MT (models/model.py:529-684,
 * :709-750, :895-1167; selected by --model_name, experiment.py:317-347).  Exact fp32.
 *   cer_linear_forward : y[r,:] = act(x[r,:] W^T + b), W [out_dim][in_dim] (nn.Linear layout);
 *                        act 0 none, 1 LeakyReLU(0.01) (F.leaky_relu, model.py:680), 2 ReLU (:734).
 *                        ldx / ldy: row pitches in floats (write into a slice of a concat buffer).
 *   cer_softmax_gate   : out = softmax(gate, dim=-1) * feat        (AttentionFusion, :563-567)
 *   cer_sdpa_forward   : out[b,i,:] = softmax_j(q[b,i,:].k[b,j,:] / sqrt(dim)) v[b,j,:] -- the core of
 *                        nn.MultiheadAttention(dim, 1) (:731, :917-931) on batch-major [B][L][dim] rows
 *   cer_add_layernorm  : out = LayerNorm(x + res) (res may be NULL)  (TransformerEncoderLayer, :740-750)
 * ------------------------------------------------------------------------------------------ */
int cer_linear_forward(const float* x_dev, int64_t rows, int32_t in_dim, int32_t ldx, const float* w_dev,
                       const float* bias_dev /* or NULL */, int32_t out_dim, int32_t act, float* y_dev, int32_t ldy, void* stream);
int cer_softmax_gate(const float* gate_dev, const float* feat_dev, int64_t rows, int32_t dim, float* out_dev, void* stream);
int cer_sdpa_forward(const float* q_dev, int32_t ldq, const float* k_dev, int32_t ldk, const float* v_dev, int32_t ldv,
                     int32_t batch, int32_t len_q, int32_t len_k, int32_t dim, float* out_dev, int32_t ldo, void* stream);
/* The same attention on the tensor cores (flash-attention forward, TF32 mma with fp32 accumulate and an fp32
 * online softmax): dim 64 or 128; q / k / v 16-byte aligned with row pitches that are multiples of 4 floats.
 * Any len_q / len_k (ragged tiles are masked).  Result within ~1e-3 of cer_sdpa_forward. */
int cer_sdpa_tc_forward(const float* q_dev, int32_t ldq, const float* k_dev, int32_t ldk, const float* v_dev, int32_t ldv,
                        int32_t batch, int32_t len_q, int32_t len_k, int32_t dim, float* out_dev, int32_t ldo, void* stream);
/* y = tanh(y) in place: the output squashing of task == REGRESSION (models/model.py:523, :682, :1165). */
/* a += b over n contiguous fp32 values (where the gradients of two branches meet) */
int cer_add_inplace(float* a_dev, const float* b_dev, int64_t n, void* stream);
int cer_tanh_inplace(float* y_dev, int64_t n, void* stream);
int cer_add_layernorm(const float* x_dev, const float* res_dev, int64_t rows, int32_t dim, const float* gamma_dev,
                      const float* beta_dev, float eps, float* out_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * Window stitching.   Replaces the sum / overlap-count / divide of
 * Trainer.inference_forward_windows (trainer.py:864-890) on device.
 * win_logits: fp32 [n_windows][win_len][n_out]; win_start: int32 [n_windows] first frame of each
 * window; out: fp32 [length][n_out] = mean over the windows covering each frame.
 * ------------------------------------------------------------------------------------------ */
int cer_stitch_windows(const float* win_logits_dev, const int32_t* win_start_dev, int32_t n_windows,
                       int32_t win_len, int32_t n_out, int64_t length, float* out_dev, void* stream);

/* Video-level decision rules.   Replaces format_trg_pred_video (metrics.py:88-145) for one video:
 * logits_dev fp32 [length][n_cls] (the stitched per-frame logits); out_dev int32[3] = FRAMES_VOTE,
 * FRAMES_AVG_LOGITS, FRAMES_AVG_PROBS.  ignore_last_class drops the 'Other' class first (:118-119). */
int cer_video_vote(const float* logits_dev, int64_t length, int32_t n_cls, int32_t ignore_last_class, int32_t* out_dev,
                   void* stream);

/* ------------------------------------------------------------------------------------------
 * Streaming LFAN head (streaming.StreamSession).   Advances n live streams by c frames per step
 * through the unchanged TCN (cer_tcn_block_tc_forward) and fusion (cer_fusion_head_forward)
 * kernels; these calls hold the per-stream state around them.  A step is a fixed sequence of
 * launches: the host writes one table of n * n_slots entries ([n][n_slots], each stream's active
 * windows first, in start order) and copies it to the device once.
 *
 * Per stream the session keeps, for a k = 5 LFAN (halo h_b = 4 * 2^b, ring rows R_b = 2 h_b):
 *   TCN rings   n_slots * 2 * sum_b R_b * C_in_pad(b) floats per modality (two halves, see stream.cu)
 *   logit ring  n_lslots * W * n_out floats     (the last W frames of each window's logits)
 *   input ring  W * D_m floats per modality     (the last W frames of each block-0 input)
 * With W = 300, H = 200, c <= 101 (n_slots = 2, n_lslots = 3), n_out = 7 and video / vggish / bert
 * TCNs of 512 -> [512,256,256,128], 128 -> [32,32,32,32], 768 -> [512,256,256,128] this comes to
 * 3.00 MB per stream (2.63 MB with synthetic.TCN_CHANNELS); the input rings are 1.69 MB of it.
 * streaming.StreamSession.state_bytes() computes it for a given model.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t sid;      /* persistent stream slot: row of every ring */
  int32_t slot;     /* TCN ring slot of the window: window index mod n_slots */
  int32_t lslot;    /* logit ring slot of the window: window index mod n_lslots */
  int32_t start;    /* first frame of the window, in the stream's own frames */
  int32_t t_now;    /* frames of the stream before this step */
  int32_t parity;   /* TCN ring half read this step; the other half is written */
  int32_t active;   /* 0: padding entry (staged as zeros, nothing written back) */
  int32_t reserved;
} cer_stream_entry;

/* One TemporalBlock's staged input: staged [n_entries][ring_rows + chunk][c_pad] fp32, rows of
 * frames max(start, t_now - ring_rows) + r.  Chunk rows come from src: src_len == 0: the chunk
 * input [n_entries / n_slots][chunk][src_dim] (channels zero-padded to c_pad); else the previous
 * block's output [n_entries][src_len][src_dim] staged with src_ring_rows (src_len = src_ring_rows
 * + chunk).  Earlier rows come from ring [streams][n_slots][2][ring_rows][c_pad], whose other half
 * receives the last ring_rows rows. */
int cer_stream_stage(const cer_stream_entry* table_dev, int32_t n_entries, int32_t n_slots, int32_t chunk,
                     int32_t ring_rows, int32_t c_pad, const float* src_dev, int32_t src_dim, int32_t src_len,
                     int32_t src_ring_rows, float* ring_dev, float* staged_dev, void* stream);
/* The chunk rows of the last block's output [n_entries][src_ring_rows + chunk][dim] ->
 * dst [n_entries][chunk][dim] (rows before a window's start, and inactive entries, are zero). */
int cer_stream_gather(const cer_stream_entry* table_dev, int32_t n_entries, int32_t chunk, const float* src_dev,
                      int32_t src_ring_rows, int32_t dim, float* dst_dev, void* stream);
/* win_logits [n_streams * n_slots][chunk][n_out] -> out [n_streams][chunk][n_out]: per frame the
 * mean over the windows covering it, summed in start order (the arithmetic of cer_stitch_windows);
 * each window's logits also go to logit_ring [streams][n_lslots][window_length][n_out] at its
 * window-relative row. */
int cer_stream_average(const cer_stream_entry* table_dev, int32_t n_streams, int32_t n_slots, int32_t chunk,
                       int32_t window_length, int32_t n_out, const float* win_logits_dev, float* out_dev,
                       float* logit_ring_dev, int32_t n_lslots, void* stream);
/* The chunk input src [n_streams][chunk][dim] -> ring [streams][window_length][dim] at row
 * frame mod window_length. */
int cer_stream_retain(const cer_stream_entry* table_dev, int32_t n_streams, int32_t n_slots, int32_t chunk,
                      const float* src_dev, int32_t dim, int32_t window_length, float* ring_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CER_B200_H_ */
