/*
 * libw2s_b200 - C ABI of the B200-native wav2sleep forward path.
 *
 * The reference (joncarter1/wav2sleep) has no FFI: its seam is the Python class contract of
 * wav2sleep.models.wav2sleep.Wav2Sleep (models/wav2sleep.py:16-80).  This header is the boundary a binding
 * (ctypes / cffi / pybind) attaches to; every entry point cites the reference code it replaces.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch types.
 *   - every pointer is a DEVICE pointer unless stated otherwise; descriptors (structs) live on the host.
 *   - functions never allocate device memory and never synchronise: the caller passes workspaces sized by
 *     the matching *_workspace_bytes() call and a cudaStream_t (as void*; NULL = legacy default stream).
 *   - return value 0 = ok, non-zero = error; w2s_last_error() gives a thread-local message.
 *   - activations are fp16, channels-last ([B, L, C]); accumulation and statistics are fp32.
 */
#ifndef W2S_B200_H_
#define W2S_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define W2S_MAX_BLOCKS 12
#define W2S_MAX_MIXER_LAYERS 8
#define W2S_MAX_SIGNALS 4
#define W2S_MAX_SEQ_BLOCKS 4
#define W2S_MAX_DILATIONS 8

/* ABI version of this header; bumped on any struct change. */
int w2s_abi_version(void);
/* Thread-local message of the last failing call ("" if none). */
const char* w2s_last_error(void);

/* ---------------------------------------------------------------------------------------------------------
 * Weight packing (host passes fp32 parameters exactly as they sit in the reference state_dict).
 * ------------------------------------------------------------------------------------------------------- */

/* nn.Conv1d weight [cout, cin, taps] fp32 -> fp16 UMMA operand layout [taps][cin/8][cout][8].
 * Also used for nn.Linear(4*C -> F) of SignalEncoder (models/wav2sleep.py:230,264) by viewing its
 * weight [F, 4*C] as [F, taps=4, C] -> pass taps_major = 1 (input index = tap*cin + c). */
int w2s_pack_conv_weight(const float* w, int cout, int cin, int taps, int taps_major, int split, void* out_fp16,
                         void* stream);  /* split: 0 = fp16, 1 = fp16 hi block + lo block, 2 = bf16 (measurement hook) */
size_t w2s_packed_conv_weight_bytes(int cout, int cin, int taps, int split);
/* 1 if the (cin, cout) encoder conv kernels carry operands as fp16 hi + fp16 lo pairs by default; their weights must
 * then be packed with split = 1 (hi block followed by lo block, twice the bytes).  True for cin <= 16 and cout <= 16. */
int w2s_conv_uses_split(int cin, int cout);
/* The same question for conv (cin -> cout) of encoder block `block` under the storage policy wide_blocks (see
 * w2s_encoder_desc): the wide 64-channel blocks of deep encoders carry split operands as well. */
int w2s_encoder_conv_split(int wide_blocks, int block, int cin, int cout);

/* Batched re-packing (one launch for every weight of a model, used after each optimizer step).  jobs: DEVICE array.
 * kind 0: packed[n][c][t] = w[n*sn + c*sc + t*st] (element strides, may be negative: flipped / transposed / sliced views
 * of the fp32 parameters) -> UMMA conv layout of w2s_pack_conv_weight (split: hi block then lo block).
 * kind 1: linear weight element (row, col) = w[row*sn + col*sc], cout = rows n, cin = columns k -> w2s_pack_linear_frag
 * order.  max_elems = largest cout*cin*taps among the jobs. */
typedef struct w2s_pack_job {
  const float* w;
  void* out;
  int32_t kind, cout, cin, taps;
  int64_t sn, sc, st;
  int32_t split, reserved;
} w2s_pack_job;
int w2s_pack_batch(const w2s_pack_job* jobs_device, int n_jobs, int max_elems, void* stream);

/* nn.Linear weight [n, k] fp32 -> fp16 mma.sync B-fragment order [n/8][k/16][32 lanes][4] (epoch mixer). */
int w2s_pack_linear_frag(const float* w, int n, int k, void* out_fp16, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * One generic implicit-GEMM conv layer (kernel-level entry, used by the tests and by the stage calls below).
 * Replaces ConvLayer1D.forward (models/blocks.py:173-186) + the consumer-side InstanceNorm/GELU of its input.
 * ------------------------------------------------------------------------------------------------------- */
enum { W2S_PRO_NONE = 0, W2S_PRO_NORM = 1, W2S_PRO_NORM_RES = 2, W2S_PRO_FIR = 3, W2S_PRO_NORM_RES_X = 4, W2S_PRO_DNORM = 5 };
enum { W2S_EPI_STATS = 0, W2S_EPI_BIAS_GELU = 1, W2S_EPI_LN_GELU = 2, W2S_EPI_LN_GELU_RES = 3, W2S_EPI_PLAIN = 4,
       W2S_EPI_ACT_BWD = 5 };

typedef struct w2s_conv_call {
  int32_t cin, cout, taps, stride, dilation, pad;
  int32_t prologue, epilogue, has_ds;
  int32_t B, L_in, L_out;
  const void* in;         /* fp16 [B, L_in, cin] */
  const void* in_res;     /* fp16 [B, L_in, cin]      (W2S_PRO_NORM_RES) */
  const double* in_stats; /* [B, cin, 2] sum, sumsq   (W2S_PRO_NORM*)    */
  const void* w;          /* packed fp16 */
  const void* w_ds;       /* packed fp16 1x1          (has_ds) */
  void* out;              /* fp16 [B, L_out, cout] */
  void* out_ds;           /* fp16 [B, L_out/2, cout]  (has_ds; row j: 1x1 branch of row 2j, L_out/2 rounded down) */
  double* out_stats;      /* [B, cout, 2], pre-zeroed (W2S_EPI_STATS) */
  const uint8_t* row_mask;/* [B] or NULL */
  const float* bias;      /* [cout] (W2S_EPI_BIAS_GELU) */
  const float* ln_w;      /* [cout] (W2S_EPI_LN_*) */
  const float* ln_b;
  const void* res;        /* fp16 [B, L_out, cout] (W2S_EPI_LN_GELU_RES) */
  const float* head_w;    /* [n_classes, cout] or NULL */
  const float* head_b;
  float* logits;          /* [B, L_out, n_classes] */
  int32_t n_classes;
  float in_eps, ln_eps;
  /* W2S_EPI_PLAIN: out = acc (+ bias) (+ res), written to row o*out_stride + out_offset of a sample of out_rows
   * rows (0, 0, 0 = dense: stride 1, offset 0, out_rows = L_out); res uses the same indexing. */
  int32_t out_stride, out_offset, out_rows;
  /* block-0 fusion (W2S_PRO_FIR: the input is conv1(x) recomputed from the raw signal; W2S_PRO_NORM_RES_X: the residual
   * branch is w_first_ds * x[2i]); x_raw fp32 [B, T_raw] with T_raw a multiple of 4, w_first fp32 [16,3],
   * w_first_ds fp32 [16]. */
  const float* x_raw;
  const float* w_first;
  const float* w_first_ds;
  int32_t T_raw;
  /* wide storage (encoder EPI_STATS convs with cin, cout <= 64 only): in / in_res, resp. out / out_ds, are fp32
   * instead of fp16 tensors of the same shape. */
  int32_t in_wide, out_wide;
  /* 1: operands are fp16 hi + lo pairs although w2s_conv_uses_split(cin, cout) is 0 (weights packed with split = 1);
   * built for the wide-storage 64-channel encoder kernels only. */
  int32_t force_split;
  /* W2S_EPI_ACT_BWD (training): data-gradient conv fused with the backward through the activation of the layer that
   * produced this conv's input: da = acc (+ res); with x_hat = InstanceNorm(act_y) [block outputs: s = GELU(x_hat) +
   * act_r, ds = da GELU'(s), act_dr = ds] out = d(x_hat) = ds GELU'(x_hat); act_a = the activated tensor (may be
   * NULL); out_stats[B, cout, 2] += (sum d(x_hat), sum d(x_hat) x_hat) (fp64, caller-zeroed).  All [B, L_out, cout]. */
  const void* act_y;
  const void* act_r;
  const double* act_stats;
  void* act_a;
  void* act_dr;
  float act_eps;
  /* W2S_PRO_DNORM (training, data-gradient convs; ABI v3): the conv input is dy = InstanceNorm-backward of `in` =
   * d(x_hat) with `in_res` = the layer's stored pre-norm output y, `in_stats` = its forward sums and dn_sums =
   * [B, cin, 2] (sum d(x_hat), sum d(x_hat) x_hat), computed on the way into shared memory; every tile also writes the
   * dy rows it owns to dn_out [B, L_in, cin] (operand of the weight gradient).  dn_upsample = 1: the layer was a
   * stride-2 conv (in / in_res have L_in / 2 rows): row i of the conv input is source row i / 2 for even i and zero for
   * odd i, dn_out is written zero-stuffed.  Replaces a separate w2s_enc_norm_bwd pass. */
  const double* dn_sums;
  void* dn_out;
  int32_t dn_upsample;
} w2s_conv_call;

int w2s_conv1d_fwd(const w2s_conv_call* call, void* stream);
/* Two calls of identical shape and configuration in ONE launch (w2s_encoder_fwd_pair's stream / Linear kernels).
 * Fails, launching nothing, if the pair has no paired kernel. */
int w2s_conv1d_fwd_pair(const w2s_conv_call* c0, const w2s_conv_call* c1, void* stream);  /* ABI v11 */
/* ---------------------------------------------------------------------------------------------------------
 * Input staging (SURVEY 8f N1).  Replaces ParquetDataset._zscore_normalize (data/dataset.py:76-87) and the -inf fill
 * of missing signals (:170-173) for a batch of raw nights already copied to the device:
 *   out[b] = (raw[b] - mean_b) / max(std_b, 1e-6)   (std unbiased as torch.std; nights holding a non-finite sample are
 *   passed through unchanged; nights with present[b] == 0 become rows of -inf).
 * raw: [B, T] of raw_dtype 0 = fp32, 1 = fp16, 2 = int16 (ADC counts); out: fp32 [B, T]; ws: [B, 3] doubles of scratch
 * (zeroed by the call; holds sum, sumsq, non-finite flag afterwards); T % 4 == 0.
 * ------------------------------------------------------------------------------------------------------- */
int w2s_stage_zscore(const void* raw, int raw_dtype, float* out, const uint8_t* present, double* ws, int B, int64_t T,
                     void* stream);

/* Profiling aid: with W2S_DEBUG_FLAGS & 64 in the environment, CTA 0 of the streaming conv kernel records %globaltimer
 * (ns) at its pipeline milestones and every CTA its entry / exit time; this copies the 16 milestone slots and
 * (optionally) the [512][2] entry/exit table of the last launch to the host (synchronises). */
int w2s_debug_timestamps(uint64_t* out16, uint64_t* cta1024);
/* Kernel selection for the encoder convs (testing / A-B measurement): 0 = auto (persistent warp-specialised
 * streaming kernel, conv_stream.cuh), 1 = tile-per-CTA kernel only (conv_igemm.cuh).  Same results either way.
 * 3 = measurement hook: tile-per-CTA kernel with BF16 MMA operands (k3 32->32 / 64->64 / 128->128 W2S_EPI_STATS convs
 * without the 1x1 branch only; weights packed with split = 2 = one block of bf16) - the hardware evidence behind the
 * fp16-over-bf16 operand decision (DESIGN.md "Numerics"); never used by the model path. */
int w2s_set_conv_impl(int impl);

/* ---------------------------------------------------------------------------------------------------------
 * Stage 1: signal encoder.  Replaces SignalEncoders.forward for one signal (models/wav2sleep.py:146-161)
 * = SignalEncoder.forward non-causal branch (:235-267) = Sequential(ConvBlock1D) (models/blocks.py:57-71)
 * with whole-night InstanceNorm1d(eps=1e-2) (models/utils.py:89-92) + Linear(4C->F) + GELU.
 * ------------------------------------------------------------------------------------------------------- */
typedef struct w2s_encoder_desc {
  int32_t n_blocks;                         /* log2(samples_per_epoch) - 2 */
  int32_t channels[W2S_MAX_BLOCKS];         /* out channels of block i: min(16 * 2^(i/2), 128) */
  int32_t feature_dim;                      /* 128 */
  float norm_eps;                           /* 1e-2 */
  const float* w_first;                     /* fp32 [16, 3]   cnn.0.conv1.conv.weight */
  const float* w_first_ds;                  /* fp32 [16]      cnn.0.downsample.weight */
  const void* w_conv[W2S_MAX_BLOCKS][3];    /* packed fp16 conv1..conv3 ([0][0] unused) */
  const void* w_ds[W2S_MAX_BLOCKS];         /* packed fp16 downsample ([0] unused) */
  const void* w_lin;                        /* packed fp16 linear.weight as taps=4 */
  const float* b_lin;                       /* fp32 [feature_dim] */
  /* inference only: the conv outputs of the first wide_blocks blocks are stored as fp32 instead of fp16 (allowed for
   * blocks with <= 64 channels: 2, 4 or 6, < n_blocks) and their convs carry split (hi + lo) operands.  0 = all fp16.
   * Deep stacks (EOG, 10 blocks) need it to meet the parity gates; it doubles the bytes of those layers. */
  int32_t wide_blocks;
} w2s_encoder_desc;

/* keep_activations = 0: inference, tensors rotate through a few slots; 1: every layer output is kept
 * (layout = w2s_encoder_layout) for a backward pass. */
size_t w2s_encoder_workspace_bytes(const w2s_encoder_desc* d, int B, int64_t T, int keep_activations);

/* Byte offsets of the tensors kept by keep_activations = 1, 7 per block: sum/sumsq of conv1, conv2, conv3 outputs
 * (fp64 [B, C, 2] each), y1 [B, L, C], r [B, L/2, C], y2 [B, L, C], y3 [B, L/2, C] (fp16).  offsets: host int64[7*n_blocks]. */
int w2s_encoder_layout(const w2s_encoder_desc* d, int B, int64_t T, int64_t* offsets);

/* x: fp32 [B, T] raw (z-scored) signal, rows of -inf = missing signal (data/dataset.py:170-173).
 * z_out: fp16 [B, T / samples_per_epoch, feature_dim]; rows of masked samples are left untouched.
 * row_mask: [B] written with 1 for missing samples. */
int w2s_encoder_fwd(const w2s_encoder_desc* d, const float* x, int B, int64_t T, void* workspace,
                    size_t workspace_bytes, int keep_activations, void* z_out, uint8_t* row_mask, void* stream);

/* Two encoders of the SAME architecture (e.g. ECG + PPG, ABD + THX: SignalEncoders builds one SignalEncoder per
 * signal from one set of constructor arguments, models/wav2sleep.py:117-133) on inputs of the same shape: every
 * encoder conv layer of the two runs in ONE launch, half of the grid each (results identical to two w2s_encoder_fwd
 * calls).  Each encoder has its own workspace of workspace_bytes.  Different architectures fall back to two plain
 * forwards in stream order.  (ABI v4) */
int w2s_encoder_fwd_pair(const w2s_encoder_desc* d0, const float* x0, void* workspace0, void* z_out0, uint8_t* row_mask0,
                         const w2s_encoder_desc* d1, const float* x1, void* workspace1, void* z_out1, uint8_t* row_mask1,
                         int B, int64_t T, size_t workspace_bytes, int keep_activations, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Stage 2: epoch mixer.  Replaces MultiModalAttentionEmbedder.forward (models/wav2sleep.py:301-346).
 * ------------------------------------------------------------------------------------------------------- */
typedef struct w2s_mixer_layer {
  const void* in_w;   /* frag-packed in_proj_weight [384,128] */
  const void* out_w;  /* frag-packed out_proj.weight [128,128] */
  const void* ff1_w;  /* frag-packed linear1.weight [512,128] */
  const void* ff2_w;  /* frag-packed linear2.weight [128,512] */
  const float *in_b, *out_b, *ff1_b, *ff2_b;
  const float *ln1_w, *ln1_b, *ln2_w, *ln2_b;
} w2s_mixer_layer;

typedef struct w2s_mixer_desc {
  int32_t n_layers;
  int32_t feature_dim; /* 128 */
  int32_t n_heads;     /* 8   */
  int32_t dim_ff;      /* 512 */
  float ln_eps;        /* 1e-5 */
  const float* cls;    /* fp32 [128] = register_tokens[0,0,:,0] */
  w2s_mixer_layer layer[W2S_MAX_MIXER_LAYERS];
} w2s_mixer_desc;

/* z[i]: fp16 [B*S, 128] features of signal i (signals sorted by name, wav2sleep.py:311);
 * row_mask[i]: [B] 1 = signal i missing for that sample (may be NULL = all present);
 * out: fp16 [B*S, 128] CLS token after the last layer. */
int w2s_epoch_mixer_fwd(const w2s_mixer_desc* d, const void* const* z, const uint8_t* const* row_mask, int n_signals,
                        int B, int S, void* out, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Stage 3: sequence mixer + classifier.  Replaces SequenceCNN.forward (models/wav2sleep.py:379-390) =
 * DilatedConvBlock x n (models/blocks.py:115-126) with ConvLayerNorm (models/utils.py:9-23) and
 * Wav2Sleep.classifier (models/wav2sleep.py:41,66).
 * ------------------------------------------------------------------------------------------------------- */
typedef struct w2s_seq_desc {
  int32_t n_blocks;      /* num_layers (2) */
  int32_t n_dilations;   /* 6 -> dilations 1..32 */
  int32_t kernel_size;   /* 7 */
  int32_t feature_dim;   /* 128 */
  int32_t n_classes;
  float ln_eps;          /* 1e-5 */
  const void* w[W2S_MAX_SEQ_BLOCKS][W2S_MAX_DILATIONS];     /* packed fp16 conv weights */
  const float* ln_w[W2S_MAX_SEQ_BLOCKS][W2S_MAX_DILATIONS]; /* fp32 [128] */
  const float* ln_b[W2S_MAX_SEQ_BLOCKS][W2S_MAX_DILATIONS];
  const float* head_w;   /* fp32 [n_classes, 128] classifier.weight */
  const float* head_b;   /* fp32 [n_classes] */
} w2s_seq_desc;

size_t w2s_seqmixer_workspace_bytes(const w2s_seq_desc* d, int B, int S, int keep_activations);

/* x: fp16 [B, S, 128] epoch-mixer output; feat_out: fp16 [B, S, 128] (may be NULL -> workspace);
 * logits: fp32 [B, S, n_classes]. */
int w2s_seqmixer_head_fwd(const w2s_seq_desc* d, const void* x, int B, int S, void* workspace, size_t workspace_bytes,
                          int keep_activations, void* feat_out, float* logits, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Training path (SURVEY section 8, row a-11): kernel-level entry points; wav2sleep_b200/training.py strings them
 * together into forward-with-saved-activations, backward, loss and optimizer step.  All tensors fp16 channels-last
 * unless noted; gradients of parameters are fp32 and ACCUMULATED (+=) into caller-zeroed buffers.
 * ------------------------------------------------------------------------------------------------------- */
/* C[m*ldc_m + n*ldc_n + t*ldc_t] += scale * sum_{b,l} X[b,l,m] * Y[b, l*y_stride + y_offset + t*tap_stride, n], t < taps
 * (weight gradients of nn.Linear (taps 1) and of all taps of an nn.Conv1d in one launch; for taps = 3, unit tap stride
 * and M, N <= 64, X and Y are read once for all taps).
 * Built for the (M,N) pairs of the model: (16,16) (32,16) (32,32) (64,32) (64,64) (128,64) (128,128). */
int w2s_gemm_tn(const void* X, const void* Y, float* C, int M, int N, int taps, int tap_stride, int B, int LX, int LY,
                int y_stride, int y_offset, long long ldc_m, long long ldc_n, long long ldc_t, float scale,
                const uint8_t* row_mask, void* stream);
/* a = GELU(InstanceNorm(y)) [then GELU(a + r)]: re-materialises the activated input of a conv (models/blocks.py:57-71). */
int w2s_enc_act_fwd(const void* y, const void* r, const double* stats, void* a, const uint8_t* row_mask, int B, int L, int C,
                    float eps, void* stream);
/* backward through GELU (and the block's residual add + GELU when r != NULL); writes d(x_hat), dr and accumulates the
 * two whole-night reductions of the InstanceNorm backward into sums[B, C, 2] (fp64, caller-zeroed).  a_out != NULL: also
 * writes the activated tensor itself (= w2s_enc_act_fwd's output) for the weight gradient of the consuming conv. */
int w2s_enc_act_bwd(const void* dout, const void* y, const void* r, const double* stats, void* dxh, void* dr, double* sums,
                    void* a_out, const uint8_t* row_mask, int B, int L, int C, float eps, void* stream);
/* dy = rstd * (dxh - mean(dxh) - x_hat * mean(dxh * x_hat)); upsample = 1 writes row 2l of a [B, 2L, C] tensor and zeros to
 * row 2l+1 (rows of masked samples are not touched). */
int w2s_enc_norm_bwd(const void* dxh, const void* y, const double* stats, const double* sums, void* dy,
                     const uint8_t* row_mask, int B, int L, int C, int upsample, float eps, void* stream);
/* weight gradients of the Cin = 1 layers of block 0 (conv1 [16,1,3] and downsample [16,1,1]), accumulated times scale. */
int w2s_first_conv_wgrad(const float* x, const void* dy1, const void* dr, float* dw1, float* dwds, const uint8_t* row_mask,
                         int B, int T, float scale, void* stream);
/* data gradient of the same two layers into the raw fp32 signal (input attribution; ABI v7):
 *   dx[b, t] = scale * (sum_c sum_k w1[c, k] dy1[b, t+1-k, c] + [t even] sum_c wds[c] dr[b, t/2, c]),
 * out-of-range dy1 rows read as 0; dx = 0 where x is non-finite and on rows with row_mask[b] != 0.  T even. */
int w2s_first_conv_dgrad(const float* x, const void* dy1, const void* dr, const float* w1, const float* wds,
                         const uint8_t* row_mask, float* dx, int B, int T, float scale, void* stream);
/* LayerNorm over 128 features per row (+GELU, + residual add + GELU): nn.LayerNorm / ConvLayerNorm (models/utils.py:9-23). */
int w2s_row_ln_fwd(const void* x, const void* res, const float* g, const float* b, void* out, long long rows, int gelu,
                   float eps, void* stream);
/* dg / db are accumulated times gscale (the inverse loss scale, see below); both NULL: not computed (frozen parameters, ABI v7). */
int w2s_row_ln_bwd(const void* x, const void* res, const float* g, const float* b, const void* dout, const void* dadd,
                   void* dx, void* ds, float* dg, float* db, long long rows, int gelu, float eps, float gscale,
                   void* stream);
int w2s_gelu_fwd(const void* pre, void* out, long long n, void* stream);
int w2s_gelu_bwd(const void* pre, const void* dout, void* din, long long n, void* stream);
/* out[c] += scale * sum over rows r of x[(r*row_stride + row_offset), c]  (bias gradients), C <= 128. */
int w2s_colsum(const void* x, float* out, long long rows, int C, int row_stride, int row_offset, const uint8_t* row_mask,
               long long rows_per_sample, float scale, void* stream);
/* nn.Dropout of the training path (nn.TransformerEncoderLayer dropout / dropout1 / dropout2, DilatedConvBlock.dropout,
 * models/blocks.py:111,123): out[i] = (keep(seed, site, i) ? x[i] / (1 - p) : 0) + (res ? res[i] : 0) over n fp16
 * elements (n % 8 == 0).  keep() is a counter-based hash of (seed, site, i), so calling it again on a gradient with the
 * same (seed, site) is the backward.  mask_out != NULL: only write the n keep decisions (0/1) there (test hook). */
int w2s_dropout(const void* x, const void* res, void* out, uint8_t* mask_out, int64_t n, float p, uint64_t seed,
                uint32_t site, void* stream);
/* 8-head attention over the D <= 5 tokens of each epoch; q,k,v,o: [N, D, 128]; key_mask [N, D] (1 = masked key).
 * drop_p > 0: dropout on the attention weights (as nn.MultiheadAttention in training), element index
 * ((n * 8 + head) * D + query) * D + key of dropout site `site`. */
int w2s_attn_fwd(const void* q, const void* k, const void* v, void* o, const uint8_t* key_mask, int N, int D, float drop_p,
                 uint64_t seed, uint32_t site, void* stream);
int w2s_attn_bwd(const void* q, const void* k, const void* v, const void* dout, void* dq, void* dk, void* dv,
                 const uint8_t* key_mask, int N, int D, float drop_p, uint64_t seed, uint32_t site, void* stream);
/* token tensor [N, 1+n_sig, 128] = [cls, z_0[n], ...] (zeros + key mask for missing signals) and its backward (dcls may be
 * NULL: the CLS gradient is not computed, ABI v7). */
int w2s_tokens_fwd(const void* const* z, const uint8_t* const* row_mask, const float* cls, void* tokens, uint8_t* key_mask,
                   int N, int S, int n_sig, void* stream);
int w2s_tokens_bwd(const void* dtokens, void* const* dz, const uint8_t* const* row_mask, float* dcls, int N, int S, int n_sig,
                   float cls_scale, void* stream);
/* out[n] = in[n*stride + offset] (scatter = 0) or out[n*stride + offset] = in[n] (scatter = 1); rows of 128 fp16. */
int w2s_rows_gather(const void* in, void* out, long long n_rows, int stride, int offset, int scatter, void* stream);
/* classifier forward, CrossEntropyLoss(mean, ignore_index) forward+backward, classifier backward. */
int w2s_head_fwd(const void* feat, const float* w, const float* b, float* logits, long long N, int C, void* stream);
int w2s_ce_fwd_bwd(const float* logits, const long long* labels, long long N, int C, long long ignore_index, double* scratch2,
                   float* loss, float* dlogits, void* stream);
/* LOSS SCALING of the backward pass.  Activation gradients are stored in fp16; with the mean cross entropy over B*S
 * epochs they are ~1e-7 at B*S = 19 200 (below fp16's normal range), so the backward runs on gradients multiplied by a
 * power of two: w2s_head_bwd writes dfeat = dfeat_scale * dlogits W (dw, db stay unscaled), every later kernel is
 * linear in the incoming gradient, and every kernel that accumulates a PARAMETER gradient multiplies by the inverse
 * (w2s_gemm_tn scale, w2s_colsum scale, w2s_row_ln_bwd gscale, w2s_first_conv_wgrad scale, w2s_tokens_bwd cls_scale),
 * so fp32 parameter gradients come out unscaled.  Reference numerics being matched: fp32 autograd
 * (scripts/config/training/main.yaml:16 `precision: 32-true`).  dw / db may be NULL (not computed; ABI v7). */
int w2s_head_bwd(const void* feat, const float* w, const float* dlogits, void* dfeat, float* dw, float* db, long long N, int C,
                 float dfeat_scale, void* stream);
/* out += sum g^2 (fp64); fused global-norm clip (torch clip_grad_norm_) + AdamW step on flat fp32 buffers.
 * ema != NULL: the same pass also updates ema = ema_decay * ema + (1 - ema_decay) * p_new, the per-batch update of the
 * reference's EMACallback (trainer/callbacks.py:54-66, SURVEY 8f N4). */
int w2s_sumsq(const float* g, long long n, double* out, void* stream);
/* *out = max |g[i]| (fp32; the call zeroes *out first; NaN if any g[i] is NaN).  Picks the loss scale of a backward
 * whose incoming gradient is not a mean cross entropy (input attribution; ABI v7). */
int w2s_absmax(const float* g, long long n, float* out, void* stream);
/* Integrated gradients (ABI v10).  out [K * B, T] = the K interpolated batches out[k, b, t] = x0 + alphas[k] * (x - x0)
 * (alphas: K device floats; x0 NULL: zero baseline).  A non-finite x[b, t] is copied unchanged onto every step, so a
 * missing (-inf) row stays missing and w2s_gen_conv / w2s_first_conv_dgrad keep reading such samples as 0. */
int w2s_ig_path_inputs(const float* x, const float* x0, const float* alphas, int K, int B, int T, float* out, void* stream);
/* attr [B, T] = (first ? 0 : attr) + (x - x0) * sum_k weights[k] * grads[k, b, t] (grads [K * B, T], weights K device
 * floats, x0 NULL: zero baseline); exactly 0 where x is non-finite.  Each step's term is added to the fp32 running sum
 * in k order, so splitting the steps over several calls (first = 0 after the first) gives bitwise the one-call sum. */
int w2s_ig_accumulate(const float* grads, const float* weights, int K, const float* x, const float* x0, int B, int T,
                      float* attr, int first, void* stream);
int w2s_adamw_step(float* p, const float* g, float* m, float* v, long long n, const double* gnorm_sq, float lr, float beta1,
                   float beta2, float eps, float weight_decay, float max_norm, float grad_scale, long long step, float* ema,
                   float ema_decay, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * General fp32 path: the NON-DEFAULT model options of the reference (SURVEY 8f N3) - causal / chunk-causal encoders
 * (models/wav2sleep.py:248-255, models/blocks.py:150-152,178-182), norms batch / layer / rms / group / auto
 * (models/utils.py:77-96), activations relu / leaky / silu / linear (utils.py:61-74), any feature_dim / nhead / dim_ff,
 * register tokens, signal embeddings, output norm, causal sequence mixer.  Dimension-generic fp32 CUDA-core kernels on
 * channels-last fp32 tensors with PyTorch weight layouts; wav2sleep_b200/general.py strings them together.  The default
 * configuration's inference and training run on the tcgen05 kernels above; its fp32 check mode
 * (Wav2Sleep.forward_fp32_check, logits within 1e-4 of the reference) runs on these kernels.
 * ------------------------------------------------------------------------------------------------------- */
enum { W2S_ACT_LINEAR = 0, W2S_ACT_RELU = 1, W2S_ACT_LEAKY = 2, W2S_ACT_GELU = 3, W2S_ACT_SILU = 4 };
enum { W2S_NORM_INSTANCE = 0, W2S_NORM_GROUP = 1, W2S_NORM_BATCH_EVAL = 2 };
/* out[b, lo, co] = bias[co] + sum_{t, ci} in[b, lo*stride - pad_left + t*dil, ci] * w[co, ci, t] (zero outside the input;
 * a causal ConvLayer1D is pad_left = (k-1)*dil, L_out = (L_in - 1) / stride + 1).  taps_major: w is [cout, taps*cin].
 * raw_inf_to_zero: `in` is the raw signal, non-finite samples read as 0. */
int w2s_gen_conv(const float* in, const float* w, const float* bias, float* out, const uint8_t* row_mask, int B, int L_in,
                 int L_out, int cin, int cout, int taps, int stride, int dil, int pad_left, int taps_major,
                 int raw_inf_to_zero, void* stream);
/* stats[b, c] = (sum, sum of squares) over L of x[b, :, c], fp64. */
int w2s_gen_stats(const float* x, double* stats, const uint8_t* row_mask, int B, int L, int C, void* stream);
/* scale / shift [B, C] of y = x * scale + shift for InstanceNorm1d, GroupNorm(groups) or eval-mode BatchNorm1d. */
int w2s_gen_norm_consts(const double* stats, const float* weight, const float* bias, const float* running_mean,
                        const float* running_var, float* scale, float* shift, int B, int C, int L, int mode, int groups,
                        float eps, void* stream);
/* out = act(in * scale[b, c] + shift[b, c] + res) (each of scale / shift / res may be NULL; per_channel: scale / shift are [C]). */
int w2s_gen_affine_act(const float* in, const float* scale, const float* shift, const float* res, float* out,
                       const uint8_t* row_mask, int B, int L, int C, int act, int per_channel, void* stream);
/* per-row LayerNorm (rms = 0) / RMSNorm (rms = 1) over C features, affine weight (+ bias), activation. */
int w2s_gen_rownorm(const float* x, const float* weight, const float* bias, float* out, long long rows, int C, int rms, int act,
                    float eps, void* stream);
/* H-head attention over the D tokens of each of N epochs; q, k, v: rows of ld >= H*hd floats ([N, D, ld], e.g. ld = 3*H*hd
 * for column slices of one fused in-projection), o: [N, D, H*hd]; key_mask [N, D] (1 = masked).  drop_p > 0: dropout on
 * the attention weights (nn.MultiheadAttention in training), keep decision of element ((n*H + h)*D + query)*D + key of
 * dropout site `site` (the generator of w2s_dropout).  drop_p = 0: no dropout.  (ABI v5: ld, drop_p, seed, site) */
int w2s_gen_attn(const float* q, const float* k, const float* v, float* o, const uint8_t* key_mask, int N, int D, int H, int hd,
                 int ld, float drop_p, uint64_t seed, uint32_t site, void* stream);

/* Backward of the general path (training of the non-default options; ABI v5).  Same conventions as the forward entry
 * points; rows of samples with row_mask[b] != 0 are skipped (their gradients stay as the caller initialised them, and they
 * add nothing to any reduction).  Parameter gradients are written (not accumulated).  The fp64 workspaces `ws` / `sums`
 * are zeroed by the call itself. */
/* din[b, li, ci] = sum over (lo, t) with lo*stride - pad_left + t*dil = li of dout[b, lo, co] * w[co, ci, t]  (gather, no
 * atomics; every case of w2s_gen_conv incl. taps_major). */
/* eval-mode BatchNorm1d: dweight = (dscale - running_mean * dshift) / sqrt(running_var + eps), dbias = dshift, all [C]
 * (the parameters behind w2s_gen_norm_consts' batch-mode scale / shift; either output may be NULL; ABI v7). */
int w2s_gen_bn_eval_bwd(const float* dscale, const float* dshift, const float* running_mean, const float* running_var,
                        float* dweight, float* dbias, int C, float eps, void* stream);
/* Train-mode BatchNorm1d statistics (ABI v8): stats[c] = fp64 (sum, sum of squares) over all rows of a [rows, C] fp32 tensor
 * (a channels-last [B, L, C] tensor is rows = B * L; stats is then what w2s_gen_norm_consts with W2S_NORM_INSTANCE, B = 1,
 * L = rows and w2s_gen_norm_bwd with B = 1, groups = C read).  Zeroes stats itself; refuses rows < 1 and C < 1. */
int w2s_gen_bn_stats(const float* x, double* stats, long long rows, int C, void* stream);
/* BatchNorm1d's running-statistics update of one training forward from those stats over n values per channel (ABI v8):
 * *num_batches_tracked += 1 (int64, on the device); f = momentum, or 1 / num_batches_tracked when momentum < 0
 * (momentum=None); running_mean = (1 - f) running_mean + f mean, running_var = (1 - f) running_var + f var n / (n - 1)
 * (unbiased variance).  fp64 arithmetic (momentum is a double, as PyTorch's Python float), fp32 buffers.  Refuses n < 2, as PyTorch does. */
int w2s_gen_bn_update_running(const double* stats, long long n, float* running_mean, float* running_var,
                              long long* num_batches_tracked, double momentum, int C, void* stream);
int w2s_gen_conv_dgrad(const float* dout, const float* w, float* din, const uint8_t* row_mask, int B, int L_in, int L_out, int cin,
                       int cout, int taps, int stride, int dil, int pad_left, int taps_major, void* stream);
/* dw[co, ci, t] = sum_{b, lo} dout * in (layout of w2s_gen_conv's w), dbias[co] = sum dout; non-finite raw samples read as 0
 * (raw_inf_to_zero).  dw or dbias may be NULL.  ws: taps*cin*cout + cout doubles. */
int w2s_gen_conv_wgrad(const float* in, const float* dout, float* dw, float* dbias, double* ws, const uint8_t* row_mask, int B,
                       int L_in, int L_out, int cin, int cout, int taps, int stride, int dil, int pad_left, int taps_major,
                       int raw_inf_to_zero, void* stream);
/* Backward of w2s_gen_affine_act: dpre = dout * act'(in * scale + shift + res); din = dpre * scale (NULL: skipped); dpre (the
 * residual gradient; NULL: skipped); sums (NULL: skipped) = fp64 (sum dpre, sum dpre * in) per [b, c] (per [c] when
 * per_channel), i.e. the shift and scale gradients. */
int w2s_gen_affine_act_bwd(const float* in, const float* scale, const float* shift, const float* res, const float* dout, float* din,
                           float* dpre, double* sums, const uint8_t* row_mask, int B, int L, int C, int act, int per_channel,
                           void* stream);
/* InstanceNorm (groups = C) / GroupNorm backward: from the forward's stats and the sums of w2s_gen_affine_act_bwd over
 * the conv output x, dx = alpha * dpre + beta * x + gamma per [b, c] (coef: workspace of B*C*3 floats); dweight / dbias
 * (NULL: skipped) of the affine GroupNorm. */
int w2s_gen_norm_bwd(const float* x, const float* dpre, const double* stats, const double* sums, const float* weight, float* coef,
                     float* dx, float* dweight, float* dbias, const uint8_t* row_mask, int B, int L, int C, int groups, float eps,
                     void* stream);
/* Backward of w2s_gen_rownorm (fused activation included): dx, and dweight / dbias (NULL: skipped) as fp64 column sums over
 * the rows (ws: 2*C doubles, needed when either is requested).  C <= 2048. */
int w2s_gen_rownorm_bwd(const float* x, const float* weight, const float* bias, const float* dout, float* dx, float* dweight,
                        float* dbias, double* ws, long long rows, int C, int rms, int act, float eps, void* stream);
/* Backward of w2s_gen_attn (same key mask, same dropout decisions): dq, dk, dv with the row stride ld of q, k, v; dout has
 * rows of H*hd.  Masked keys get dk = dv = 0. */
int w2s_gen_attn_bwd(const float* q, const float* k, const float* v, const float* dout, float* dq, float* dk, float* dv,
                     const uint8_t* key_mask, int N, int D, int H, int hd, int ld, float drop_p, uint64_t seed, uint32_t site,
                     void* stream);
/* fp32 dropout over any n < 2^32 elements: out[i] = keep(seed, site, i) ? x[i] / (1 - p) : 0, the decisions of w2s_dropout;
 * applied to the gradient it is the backward.  mask_out != NULL: only write the n keep decisions (0/1) there (test hook). */
int w2s_gen_dropout(const float* x, float* out, uint8_t* mask_out, long long n, float p, uint64_t seed, uint32_t site,
                    void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Streaming step of a causal sequence mixer (ABI v6; wav2sleep_b200/streaming.py).  Every DilatedConvBlock of a causal
 * SequenceCNN (models/blocks.py:115-126, ConvLayer1D causal :150-152, :178-182) and the classifier, for R new epochs of
 * N streams, in eval semantics (running BatchNorm statistics, no dropout), fp32.  The history of each dilated layer is a
 * ring in `ring`: layer l = b * n_dilations + j (dilation 2^j) keeps M_l = (k-1) * 2^j input rows of F floats per stream;
 * the row of epoch e is in slot e mod M_l.  A stream's state is n_blocks * (k-1) * (2^n_dilations - 1) rows of F floats,
 * its layers' rings one after the other: ring[n, off_l + slot, :] with off_l = sum of M over the layers before l.  Zero
 * rows are the causal zero padding, so a stream restarts when the caller zeroes its rows.  Parameters are read in place.
 * ------------------------------------------------------------------------------------------------------- */
#define W2S_STREAM_MAX_LAYERS 32     /* n_blocks * n_dilations */
#define W2S_STREAM_MAX_DILATIONS 16
#define W2S_STREAM_MAX_KERNEL 16
#define W2S_STREAM_MAX_FEATURES 256
enum { W2S_SEQ_NORM_NONE = 0, W2S_SEQ_NORM_BATCH = 1, W2S_SEQ_NORM_LAYER = 2, W2S_SEQ_NORM_RMS = 3 };

typedef struct w2s_gen_seq_stream_layer {
  const float* w;             /* conv.weight [F, F, k] */
  const float* bias;          /* conv.bias [F] or NULL (ConvLayer1D has one only without a norm) */
  const float* norm_w;        /* norm weight [F] or NULL (= 1) */
  const float* norm_b;        /* norm bias [F] or NULL (= 0) */
  const float* running_mean;  /* W2S_SEQ_NORM_BATCH: running statistics [F] */
  const float* running_var;
} w2s_gen_seq_stream_layer;

typedef struct w2s_gen_seq_stream_desc {
  int32_t n_blocks;      /* num_layers */
  int32_t n_dilations;   /* dilations 1, 2, .., 2^(n_dilations-1) */
  int32_t kernel_size;
  int32_t feature_dim;   /* F */
  int32_t n_classes;
  int32_t norm;          /* W2S_SEQ_NORM_* */
  int32_t act;           /* W2S_ACT_* */
  float eps;             /* of the norm */
  w2s_gen_seq_stream_layer layer[W2S_STREAM_MAX_LAYERS];
  const float* head_w;   /* classifier.weight [n_classes, F] */
  const float* head_b;   /* classifier.bias [n_classes] */
  float* ring;           /* [N, n_blocks * (k-1) * (2^n_dilations - 1), F], read and written */
} w2s_gen_seq_stream_desc;

/* x_new: [N, R, F] epoch-mixer features of epochs pos .. pos+R-1 -> logits [N, R, n_classes]; one launch, epochs in
 * order.  Limits: F <= W2S_STREAM_MAX_FEATURES, 1 <= kernel_size <= W2S_STREAM_MAX_KERNEL, n_dilations <=
 * W2S_STREAM_MAX_DILATIONS, n_blocks * n_dilations <= W2S_STREAM_MAX_LAYERS. */
int w2s_gen_seq_stream_step(const w2s_gen_seq_stream_desc* d, const float* x_new, float* logits, int N, int R, long long pos,
                            void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Measurement hooks (bench.py).  Not part of the data path.
 * ------------------------------------------------------------------------------------------------------- */
/* Number of kernels this library has launched in this process (monotonic). */
long long w2s_launch_count(void);
/* on = 1: every later launch is bracketed by CUDA events on its stream and recorded; on = 0: stop and clear. */
int w2s_profile_enable(int on);
int w2s_profile_count(void);
/* Record i: label (host buffer), elapsed ms (synchronises on the record's end event), algorithmic bytes / flops. */
int w2s_profile_get(int i, char* label, int label_cap, float* ms, double* bytes, double* flops);

/* argmax over classes (Wav2Sleep.predict, models/wav2sleep.py:69-80): logits fp32 [n, c] -> int64 [n]. */
int w2s_argmax(const float* logits, int64_t n, int n_classes, int64_t* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* W2S_B200_H_ */
