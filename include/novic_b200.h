/*
 * novic_b200 - C ABI of the B200-native NOVIC object-noun decoder hot path.
 *
 * The reference (pallgeuer/novic) has no FFI: its seam for this path is the Python class contract of
 * `embedding_decoder.PrefixedIterDecoder` (embedding_decoder.py:617-1079) selected by name at
 * infer.py:716.  `novic_b200/decoder.py` mirrors that class; its methods call the entry points below through
 * ctypes.  Each entry point names the reference function it replaces.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; `novic_last_error()` describes the failure
 *   - all pointers marked "device" are raw CUDA device pointers owned by the caller (torch tensors) and are
 *     only borrowed for the duration of the call; work is enqueued on the `stream` argument
 *     (a cudaStream_t passed as void*), calls that return a host value synchronise that stream
 *   - a handle is bound to the CUDA device that was current at novic_create(); handles are not thread-safe
 *   - token ids are int64, masks are 1-byte booleans, scores / logits are fp32 (what the reference returns)
 *   - there is no CPU fallback: without an sm_100 device every compute entry point fails
 */
#ifndef NOVIC_B200_H_
#define NOVIC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NOVIC_MAX_LAYERS 16
#define NOVIC_MAX_BEAMS 16

/* Architecture of the decoder; mirrors the constructor arguments of PrefixedIterDecoder
 * (embedding_decoder.py:43-75, :633-640) that influence the computation. */
typedef struct NovicCfg {
  int32_t embed_dim;       /* F: CLIP embedding size (embedder.embed_dim, embedding_decoder.py:86)            */
  int32_t hidden_dim;      /* E: must be 512 (kernels are specialised for config/train.yaml:256)              */
  int32_t ffn_dim;         /* K: hidden_dim * feedfwd_scale, must be 128                                      */
  int32_t num_layers;      /* L <= NOVIC_MAX_LAYERS                                                           */
  int32_t num_heads;       /* must be 8 (head dim 64)                                                         */
  int32_t prefix_len;      /* P = mlp_seq_len                                                                 */
  int32_t vocab_size;      /* V = target_config.vocab_size (rows of the tied matrix actually used)            */
  int32_t token_length;    /* Cmax = target_config.token_length                                               */
  int32_t strictly_causal; /* embedding_decoder.py:652                                                        */
  int32_t num_end_loss;    /* embedding_decoder.py:700                                                        */
  float ln_eps;            /* 1e-5                                                                            */
  float label_smoothing;   /* embedding_decoder.py:738                                                        */
} NovicCfg;

/* fp32 parameters exactly as the reference's state dict holds them (SURVEY.md section 8 row a1). */
typedef struct NovicWeights {
  const float* embed_mlp;                  /* embed_mlp.mlp.0.weight               [P*E, F]   */
  const float* tok_embed;                  /* logits_linear.weight (tied)          [>=V, E]   */
  const float* pos_embed;                  /* pos_embedding.embedding.weight       [P+Cmax-1, E] */
  const float* final_norm;                 /* transformer.norm.weight              [E]        */
  const float* in_proj[NOVIC_MAX_LAYERS];  /* ...layers.i.self_attn.in_proj_weight [3E, E]    */
  const float* out_proj[NOVIC_MAX_LAYERS]; /* ...layers.i.self_attn.out_proj.weight [E, E]    */
  const float* linear1[NOVIC_MAX_LAYERS];  /* ...layers.i.linear1.weight           [K, E]     */
  const float* linear2[NOVIC_MAX_LAYERS];  /* ...layers.i.linear2.weight           [E, K]     */
  const float* norm1[NOVIC_MAX_LAYERS];    /* ...layers.i.norm1.weight             [E]        */
  const float* norm2[NOVIC_MAX_LAYERS];    /* ...layers.i.norm2.weight             [E]        */
} NovicWeights;

/* Embedding-noise configuration; mirrors EmbeddingNoise.create (embedding_noise.py:17-41). Angles in degrees. */
typedef struct NovicNoiseCfg {
  int32_t scheme;     /* 0 GaussElem, 1 GaussVec, 2 GaussAngle, 3 UniformAngle, 4 GaussElemUniformAngle */
  int32_t embed_dim;
  float vec_norm, angle_min, angle_max, angle_std, mix_ratio;
} NovicNoiseCfg;

/* Guided decoding (embedding_decoder.py:802-813 greedy, :873-878 / :915-920 / :942-943 / :969-971 beam): the W x Cmax
 * guide_targets tensor the reference receives (built at infer.py:687-710) as a token trie in CSR form, built on the host
 * by novic_b200/guide.py.  Node 0 is the root; the ids allowed after a prefix are the token ids of its node's child
 * edges.  All three arrays are int32 device pointers borrowed for the call. */
typedef struct NovicGuide {
  const int32_t* child_off;  /* [num_nodes + 1] */
  const int32_t* child_tok;  /* [num_edges], ascending within a node */
  const int32_t* child_node; /* [num_edges] */
  int32_t num_nodes;
  int32_t num_edges;
  int32_t renorm;            /* guide_renorm: renormalise the scores over the allowed ids */
  const float* child_bias;   /* optional [num_edges] fp32, beam search only: additive score of taking each edge - the
                              * vocabulary prior -vocab_scaler * log p_vocab(token | prefix) of embedding_decoder.py:924-936
                              * (-inf: no vocabulary noun continues that way).  NULL = no prior. */
} NovicGuide;

typedef struct NovicHandle NovicHandle;

const char* novic_last_error(void);
int novic_version(void);

/* Replaces PrefixedIterDecoder.__init__ (embedding_decoder.py:633-654) for the compute side. */
int novic_create(const NovicCfg* cfg, NovicHandle** out);
int novic_destroy(NovicHandle* h);

/* Bytes of device memory novic_set_weights needs for its bf16 / packed copies. */
size_t novic_weight_bytes(const NovicHandle* h);
/* Replaces load_state_dict(...) + .to(device) (infer.py:776, :184): converts the fp32 parameters into the
 * kernels' bf16 operand layout inside `wbuf` (device, caller-owned, must outlive the handle's use). */
int novic_set_weights(NovicHandle* h, const NovicWeights* w, void* wbuf, size_t wbuf_bytes, void* stream);

/* Workspace (KV cache pages, activations, selection partials) for a call over `num_embeds` embeddings with
 * `seqs_per_embed` sequences each (beam width H, or multi-target count M, or 1) and `rows_per_seq` residual
 * rows per sequence (0 = decode: max(P, 1) rows; else P + C - 1 for teacher forcing). */
size_t novic_workspace_bytes(const NovicHandle* h, int64_t num_embeds, int32_t seqs_per_embed, int32_t rows_per_seq);

/* Replaces PrefixedIterDecoder.generate (embedding_decoder.py:779-850); guide = NULL: unguided.
 *   embed [B, F] fp32 device.  Outputs (device): tok [B, G] int64, pad [B, G] u8, score [B] fp32,
 *   nll [B] fp32 (per-sample sum of -log p over unpadded tokens, label smoothing applied), len [B] fp32
 *   (unpadded tokens per sample), logits [B, G, V] fp32 or NULL.  *T_out (host) = number of columns the
 *   reference would return (early exit when every sample has emitted the end token). G = Cmax - 1. */
int novic_generate_greedy(NovicHandle* h, const float* embed, int64_t B, float temperature, float length_alpha,
                          int64_t* tok, uint8_t* pad, float* score, float* nll, float* len, float* logits,
                          int32_t* T_out, const NovicGuide* guide, void* ws, size_t ws_bytes, void* stream);

/* The same decode without the host synchronisation: everything is enqueued on `stream` and the early-exit length is written to
 * T_dev (device int32) instead of being returned, so a serving loop can enqueue the next batch while this one runs
 * (novic_b200/serve.py).  tok / pad hold all G columns; the caller cuts them to T_dev[0] once it has read the results back.
 * The workspace may be reused by the next call on the same stream. */
int novic_generate_greedy_async(NovicHandle* h, const float* embed, int64_t B, float temperature, float length_alpha,
                                int64_t* tok, uint8_t* pad, float* score, float* nll, float* len, int32_t* T_dev,
                                const NovicGuide* guide, void* ws, size_t ws_bytes, void* stream);

/* Tail of PrefixedIterDecoder.generate (embedding_decoder.py:838-846): loss_sum = sum_b w_b * nll_b and loss_basis = sum_b w_b * len_b over
 * the per-sample vectors novic_generate_greedy returns (weight = sample_weight, NULL = 1), as one deterministic single-block reduction.
 *   out_f32x2 [2] fp32 device = {loss_sum, loss_basis}; out_i64 [1] int64 device (may be NULL) = loss_basis rounded to an integer
 *   (what the reference returns without sample weights). */
int novic_loss_totals(const float* nll, const float* len, const float* weight, int64_t n, float* out_f32x2, int64_t* out_i64, void* stream);

/* Replaces PrefixedIterDecoder.generate_beam (embedding_decoder.py:852-984); guide = NULL: unguided, no vocabulary prior.
 * With a vocabulary prior and no guide_targets the caller passes the vocabulary trie as the guide (renorm = 0) with child_bias set.
 *   Outputs (device): tok [B, H, G] int64, pad [B, H, G] u8, score [B, H] fp32 sorted descending. */
int novic_generate_beam(NovicHandle* h, const float* embed, int64_t B, int32_t H, float temperature,
                        float length_alpha, int64_t* tok, uint8_t* pad, float* score, int32_t* T_out, const NovicGuide* guide,
                        void* ws, size_t ws_bytes, void* stream);

/* Replaces PrefixedIterDecoder.forward (embedding_decoder.py:659-777) with guide_targets=None.
 *   embed [B, F]; target [A, C] int64 with A = B * M (sequences of one embedding adjacent, multi_first=False);
 *   padding [A, C] u8 or NULL; weight [A] fp32 or NULL.  T = 1 if only_pred else C.
 *   Outputs (device, each may be NULL): logits [A, T, V] fp32, pad_out [A, T] u8 (effective target padding),
 *   loss [2] fp32 = {loss_sum, loss_basis}, correct [A, T] u8. */
int novic_forward(NovicHandle* h, const float* embed, int64_t B, int32_t M, const int64_t* target,
                  const uint8_t* padding, const float* weight, int32_t C, int32_t only_pred, float* logits,
                  uint8_t* pad_out, float* loss, uint8_t* correct, void* ws, size_t ws_bytes, void* stream);

/* novic_forward with the guided correctness evaluation of embedding_decoder.py:754-760: `correct` compares the target with the arg-max
 * over the ids that continue a guide target matching the sequence's own prefix (trie built over the first C columns of guide_targets);
 * logits, padding and loss are those of the unguided forward.  only_pred is not available (the reference asserts the same).
 * mask_scratch: caller-owned device memory of at least A * C * ceil(V / 32) * 4 bytes (A = B * M). */
int novic_forward_guided(NovicHandle* h, const float* embed, int64_t B, int32_t M, const int64_t* target,
                         const uint8_t* padding, const float* weight, int32_t C, float* logits, uint8_t* pad_out, float* loss,
                         uint8_t* correct, const NovicGuide* guide, void* mask_scratch, size_t mask_bytes, void* ws, size_t ws_bytes,
                         void* stream);

/* Replaces the scoring loop of PrefixedIterDecoder.generate_all (embedding_decoder.py:1063-1072): the teacher-forced
 * log-probability of M given token sequences for each of B embeddings, without materialising logits.
 *   target [A, C] int64 and padding [A, C] u8 (may be NULL) with A = B * M, the M sequences of an embedding adjacent.
 *   score [A] fp32 (device) = sum over unpadded positions c of log softmax(logits[a, c] / temperature)[target[a, c]].
 *   guide != NULL with renorm set (guide_renorm): the softmax at position c runs over the ids that continue a guide target
 *   matching target[a, :c]; the masks are built from the first M target rows and shared by all embeddings, so `target`
 *   must repeat with period M (what generate_all passes: the same guide targets for every embedding). */
int novic_score_targets(NovicHandle* h, const float* embed, int64_t B, int32_t M, const int64_t* target, const uint8_t* padding,
                        int32_t C, float temperature, const NovicGuide* guide, float* score, void* ws, size_t ws_bytes, void* stream);

/* Replaces the forward + backward of one training batch (train.py:1270-1273: model(..., calc_loss=True, calc_correct=True,
 * only_pred=False) followed by loss.backward()); dropout as set by novic_set_dropout.  Same inputs as novic_forward (C >= 2).
 * Outputs (device): loss [2] = {loss_sum, loss_basis}; correct [A, C] u8 and pad_out [A, C] u8 (may be NULL); `grads`
 * holds fp32 device buffers shaped like the parameters of NovicWeights and receives d(loss_sum) / d(parameter)
 * (overwritten).  The caller applies the 1 / (loss_basis * accumulation) factor, gradient clipping and the optimizer,
 * exactly as train.py:1272-1286 does. */
size_t novic_train_workspace_bytes(const NovicHandle* h, int64_t B, int32_t M, int32_t C);
/* Dropout of the following novic_train_fwd_bwd calls (embedding_decoder.py:1290,:1297 input_dropout after the positional embedding;
 * nn.TransformerEncoderLayer's layer_dropout on the attention probabilities, on both residual branches and on the activated
 * feed-forward hidden rows).  Masks are a counter-based hash of (seed, layer, site, element) - the backward pass regenerates them.
 * p = 0 switches a site off (the default); pass a fresh seed per step.  Inference entry points never apply dropout. */
int novic_set_dropout(NovicHandle* h, float p_input, float p_layer, uint64_t seed);
int novic_train_fwd_bwd(NovicHandle* h, const float* embed, int64_t B, int32_t M, const int64_t* target, const uint8_t* padding,
                        const float* weight, int32_t C, float* loss, uint8_t* correct, uint8_t* pad_out, const NovicWeights* grads,
                        void* ws, size_t ws_bytes, void* stream);

/* novic_train_fwd_bwd with a completion point inside the backward pass: once the gradients of layers >= split_layer are final (layers are
 * walked from the last to the first), `split_event` (a cudaEvent_t passed as void*) is recorded on `stream`; the rest of the call only writes
 * the gradients of layers < split_layer, of the embeddings, the positions and the prefix projection.  A data-parallel step starts the
 * all-reduce of the finished part of the gradient bucket on another stream there (novic_b200/dist.py).  split_layer <= 0: no event.
 * Both entry points replay the ~280 launches of a step as CUDA graphs (two when split) cached per shape / flags / workspace / gradient
 * addresses; inputs are staged inside the workspace and the dropout seed lives in a device word, so the graphs stay valid across steps. */
int novic_train_fwd_bwd_ex(NovicHandle* h, const float* embed, int64_t B, int32_t M, const int64_t* target, const uint8_t* padding,
                           const float* weight, int32_t C, float* loss, uint8_t* correct, uint8_t* pad_out, const NovicWeights* grads,
                           void* ws, size_t ws_bytes, void* stream, int32_t split_layer, void* split_event);

/* Replaces the optimizer tail of a training step (train.py:1281-1286: clip_grad_norm_(max_norm, error_if_nonfinite) + torch.optim.AdamW.step(),
 * parameter groups of train.py:1108-1119) over ONE flat fp32 buffer each for parameters, gradients and the two moments - three launches,
 * no host synchronisation.
 *   grads: d(loss_sum) / d(parameter), n elements (n a multiple of 512), in the parameters' order.
 *   stats: device [loss_sum, loss_basis, ...] or NULL: the gradients are divided by max(loss_basis, 1) first (train.py:1272).
 *   decay_flags [n / 512] u8: chunk c receives weight decay (tensors with >= 2 dimensions).
 *   out4 (device fp32): [0] gradient norm (after the 1 / basis factor), [1] clip coefficient min(1, max_norm / (norm + 1e-6)), [2] factor
 *   applied to the raw gradients, [3] 1.0 if the norm was not finite - the update is then skipped (the reference raises at that point).
 *   max_grad_norm <= 0: no clipping (train.py:1281). */
typedef struct NovicAdamW {
  float lr, beta1, beta2, eps, weight_decay, max_grad_norm;
  int64_t step;   /* 1-based: bias corrections 1 - beta^step */
} NovicAdamW;
size_t novic_adamw_scratch_bytes(void);
int novic_adamw_step(const NovicAdamW* cfg, float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
                     const uint8_t* decay_flags, const float* stats, void* scratch, size_t scratch_bytes, float* out4, void* stream);

/* Replaces EmbeddingNoise.forward (embedding_noise.py:72-75, :90-95, :105-112, :169-172): in place on
 * embed [B, F] fp32 device; random draws come from Philox (seed, offset). */
int novic_noise_apply(const NovicNoiseCfg* cfg, float* embed, int64_t B, uint64_t seed, uint64_t offset, void* stream);
/* Deterministic variant for parity tests: the draws are supplied (device pointers, see kernels.cuh NoiseParams). */
int novic_noise_apply_predrawn(const NovicNoiseCfg* cfg, float* embed, int64_t B, const float* normals_a,
                               const float* normals_b, const float* row_a, const float* row_b, void* stream);

/* ---------------------------------------------------------------------------------------------------------------------------------
 * Image encoder in front of the decoder (SURVEY.md section 8 row f3, BASELINE config #5).  Replaces the call
 * `self.model_encode_image(images, normalize=False)` + fp32 normalise of embedders.py:759-764 for an open_clip VisionTransformer
 * (un-vendored dependency open_clip_torch==2.23, requirements.txt:8; the architecture is an assumption documented in DESIGN.md):
 * conv patch embedding without bias, class token, learned positions, ln_pre, `layers` pre-LN blocks (MultiheadAttention with biases,
 * heads of 80 channels; MLP width -> mlp_dim -> width with QuickGELU), ln_post on the class token, bias-free projection to out_dim.
 * All parameters fp32 device pointers named after open_clip's state dict (`visual.*`). */
#define NOVIC_VIT_MAX_LAYERS 48
typedef struct NovicVitCfg {
  int32_t image_size;   /* 378 */
  int32_t patch_size;   /* 14  */
  int32_t width;        /* 1280 = heads * 80 */
  int32_t layers;       /* 32 */
  int32_t heads;        /* 16 */
  int32_t mlp_dim;      /* 5120 */
  int32_t out_dim;      /* 1024 = the decoder's embed_dim */
  float ln_eps;         /* 1e-5 */
} NovicVitCfg;
typedef struct NovicVitWeights {
  const float* conv1;                 /* visual.conv1.weight                         [width, 3, patch, patch] */
  const float* class_embedding;       /* visual.class_embedding                      [width] */
  const float* positional_embedding;  /* visual.positional_embedding                 [tokens, width] */
  const float *ln_pre_w, *ln_pre_b;   /* visual.ln_pre.{weight,bias} */
  const float *ln_post_w, *ln_post_b; /* visual.ln_post.{weight,bias} */
  const float* proj;                  /* visual.proj                                 [width, out_dim] (x @ proj) */
  const float* ln1_w[NOVIC_VIT_MAX_LAYERS];      /* visual.transformer.resblocks.i.ln_1.weight */
  const float* ln1_b[NOVIC_VIT_MAX_LAYERS];
  const float* in_proj_w[NOVIC_VIT_MAX_LAYERS];  /* ...attn.in_proj_weight   [3 width, width] */
  const float* in_proj_b[NOVIC_VIT_MAX_LAYERS];  /* ...attn.in_proj_bias     [3 width] */
  const float* out_proj_w[NOVIC_VIT_MAX_LAYERS]; /* ...attn.out_proj.weight  [width, width] */
  const float* out_proj_b[NOVIC_VIT_MAX_LAYERS];
  const float* ln2_w[NOVIC_VIT_MAX_LAYERS];      /* ...ln_2.weight */
  const float* ln2_b[NOVIC_VIT_MAX_LAYERS];
  const float* fc_w[NOVIC_VIT_MAX_LAYERS];       /* ...mlp.c_fc.weight       [mlp_dim, width] */
  const float* fc_b[NOVIC_VIT_MAX_LAYERS];
  const float* cproj_w[NOVIC_VIT_MAX_LAYERS];    /* ...mlp.c_proj.weight     [width, mlp_dim] */
  const float* cproj_b[NOVIC_VIT_MAX_LAYERS];
} NovicVitWeights;
typedef struct NovicVitHandle NovicVitHandle;
int novic_vit_create(const NovicVitCfg* cfg, NovicVitHandle** out);
int novic_vit_destroy(NovicVitHandle* h);
size_t novic_vit_weight_bytes(const NovicVitHandle* h);
int novic_vit_set_weights(NovicVitHandle* h, const NovicVitWeights* w, void* wbuf, size_t wbuf_bytes, void* stream);
/* Workspace of one chunk of `images_per_chunk` images (the encoder walks a batch chunk by chunk). */
size_t novic_vit_workspace_bytes(const NovicVitHandle* h, int64_t images_per_chunk);
/* images [B, 3, image_size, image_size] fp32 device (already preprocessed) -> embed_out [B, out_dim] fp32 device, L2-normalised when
 * normalize != 0 (embedders.py:764).  The result can be handed to novic_generate_* without leaving the device. */
int novic_vit_encode(NovicVitHandle* h, const float* images, int64_t B, float* embed_out, int32_t normalize, int64_t images_per_chunk,
                     void* ws, size_t ws_bytes, void* stream);

/* The reference's default embedder, open_clip `ViT-B-16-SigLIP` (config/train.yaml:126; architecture assumed as in DESIGN.md §5d):
 * timm `vit_base_patch16_siglip_224` - patch convolution with bias, learned positions, no class token, `layers` pre-LN blocks (heads
 * of 64 channels, exact erf GELU), final LayerNorm on all tokens, MAP attention-pool head; out_dim = width.  The same structs describe
 * open_clip `ViT-SO400M-14-SigLIP` (timm `vit_so400m_patch14_siglip_224`, the F = 1152 checkpoints' embedder, assumed to be the same
 * architecture): patch 14, width 1152, 27 blocks, 16 heads of 72, mlp_dim 4304.  Accepted: width / heads = 64 or 72, width 640, 768,
 * 1024, 1152 or 1280, mlp_dim a multiple of 16 (the library pads the MLPs to whole 128-channel k-stages with zero weights; the
 * weight and workspace sizes include the padding).  novic_siglip_create and
 * novic_siglip_set_weights fill the same NovicVitHandle, so novic_vit_destroy / _weight_bytes / _workspace_bytes / _encode serve both
 * models.  All parameters fp32 device pointers named after open_clip's state dict (`visual.trunk.*`). */
typedef struct NovicSiglipCfg {
  int32_t image_size;   /* 224 */
  int32_t patch_size;   /* 16  */
  int32_t width;        /* 768 = heads * 64 = out_dim (SO400M: 1152 = heads * 72) */
  int32_t layers;       /* 12 (SO400M: 27) */
  int32_t heads;        /* 12 (SO400M: 16) */
  int32_t mlp_dim;      /* 3072 (blocks and head MLP; SO400M: 4304) */
  float ln_eps;         /* 1e-6 */
} NovicSiglipCfg;
typedef struct NovicSiglipWeights {
  const float *patch_w, *patch_b;     /* visual.trunk.patch_embed.proj.{weight,bias}  [width, 3, patch, patch], [width] */
  const float* pos_embed;             /* visual.trunk.pos_embed                       [1, tokens, width] */
  const float *norm_w, *norm_b;       /* visual.trunk.norm.{weight,bias} */
  const float* pool_latent;           /* visual.trunk.attn_pool.latent                [1, 1, width] */
  const float *pool_q_w, *pool_q_b;   /* ...attn_pool.q.{weight,bias}                 [width, width], [width] */
  const float *pool_kv_w, *pool_kv_b; /* ...attn_pool.kv.{weight,bias}                [2 width, width], [2 width] (k first) */
  const float *pool_proj_w, *pool_proj_b;   /* ...attn_pool.proj.{weight,bias}        [width, width], [width] */
  const float *pool_norm_w, *pool_norm_b;   /* ...attn_pool.norm.{weight,bias} */
  const float *pool_fc1_w, *pool_fc1_b;     /* ...attn_pool.mlp.fc1.{weight,bias}     [mlp_dim, width], [mlp_dim] */
  const float *pool_fc2_w, *pool_fc2_b;     /* ...attn_pool.mlp.fc2.{weight,bias}     [width, mlp_dim], [width] */
  const float* norm1_w[NOVIC_VIT_MAX_LAYERS];    /* visual.trunk.blocks.i.norm1.weight */
  const float* norm1_b[NOVIC_VIT_MAX_LAYERS];
  const float* qkv_w[NOVIC_VIT_MAX_LAYERS];      /* ...attn.qkv.weight       [3 width, width] */
  const float* qkv_b[NOVIC_VIT_MAX_LAYERS];      /* ...attn.qkv.bias         [3 width] */
  const float* proj_w[NOVIC_VIT_MAX_LAYERS];     /* ...attn.proj.weight      [width, width] */
  const float* proj_b[NOVIC_VIT_MAX_LAYERS];
  const float* norm2_w[NOVIC_VIT_MAX_LAYERS];    /* ...norm2.weight */
  const float* norm2_b[NOVIC_VIT_MAX_LAYERS];
  const float* fc1_w[NOVIC_VIT_MAX_LAYERS];      /* ...mlp.fc1.weight        [mlp_dim, width] */
  const float* fc1_b[NOVIC_VIT_MAX_LAYERS];
  const float* fc2_w[NOVIC_VIT_MAX_LAYERS];      /* ...mlp.fc2.weight        [width, mlp_dim] */
  const float* fc2_b[NOVIC_VIT_MAX_LAYERS];
} NovicSiglipWeights;
int novic_siglip_create(const NovicSiglipCfg* cfg, NovicVitHandle** out);
int novic_siglip_set_weights(NovicVitHandle* h, const NovicSiglipWeights* w, void* wbuf, size_t wbuf_bytes, void* stream);

/* Building-block check used by the test-suite: out[M, N] fp32 = A[M, K] (bf16) * W[N, K]^T (bf16) through the
 * same tcgen05 / TMA kernel the decoder uses.  K % 64 == 0. */
int novic_debug_gemm(const void* a_bf16, const void* w_bf16, float* out, int32_t M, int32_t N, int32_t K,
                     int32_t block_n, void* stream);

/* Building blocks of the training step's backward pass, exported for the test-suite (ragged and unaligned shapes):
 *   novic_debug_transpose_bf16: dst[c, r] = src[r, c] for a row-major bf16 [rows, cols] matrix (leading dimensions in elements);
 *   novic_debug_wgrad: dw[Mo, No] (fp32, accumulated into) += a_t[Mo, K] * b_t[No, K]^T, both operands bf16 with the contraction
 *     index contiguous and leading dimension ld (a multiple of 8) - the split-K weight-gradient GEMM;
 *   novic_debug_wgrad_splits: the split-K factor that GEMM picks for `tiles` output tiles, `kblocks` 64-wide k-blocks and `sms`
 *     CTAs (pure host arithmetic; -1 on bad arguments). */
int novic_debug_transpose_bf16(const void* src, int64_t rows, int32_t cols, int32_t ld_src, void* dst, int32_t ld_dst, void* stream);
int novic_debug_wgrad(const void* a_t, int32_t Mo, const void* b_t, int32_t No, int64_t K, int32_t ld, float* dw, void* stream);
/*   novic_debug_wgrad_mn: the same product from the UN-transposed operands, dw[Mo, No] += a[K, Mo]^T * b[K, No] (row-major bf16, leading
 *     dimensions ld_a / ld_b: multiples of 8, at least the column count rounded up to 64) - MN-major tcgen05 operand descriptors; what the
 *     training step uses (NOVIC_WGRAD_MN=0 restores the transposed copies). */
int novic_debug_wgrad_mn(const void* a, int32_t Mo, int32_t ld_a, const void* b, int32_t No, int32_t ld_b, int64_t K, float* dw, void* stream);
int32_t novic_debug_wgrad_splits(int64_t tiles, int64_t kblocks, int32_t sms);

/* Building blocks of the image encoders, exported for the test-suite: the encoder's own launch helpers on caller-owned device buffers.
 *   novic_debug_vit_gemm: acc[M, N] = a[M, K] (bf16) * w[N, K]^T (bf16), K % 128 == 0, N % 32 == 0, through epilogue
 *     epi 0 (EpiVitBias):     dst bf16 [M, ld] = act(acc + bias) (act 0 none, 1 QuickGELU, 2 erf GELU; direct: 256-bit stores from the
 *                             registers, else through the staging tile);
 *     epi 1 (EpiVitResid):    dst fp32 [*, ld]: residual mode (table NULL) dst[r] += acc + bias; patch mode dst[img * (patches + tok0) + tok0 + p]
 *                             = acc + table[(tok0 + p) * ld] + bias for GEMM row r = img * patches + p;
 *     epi 2 (EpiVitStoreF32): dst fp32 [M, N] = acc (+ bias), ld == N.
 *     bias may be NULL.  path 128 / 256 / 512 forces 128 x 128, 128 x 256 or CTA-pair 256 x 256 tiles; the persistent grid is divided by
 *     grid_div (>= 1), so that few CTAs walk many tiles.
 *   novic_debug_vit_attention: ao [nimg * T, W] bf16 = softmax(q k^T / sqrt(D)) v per (image, head) from qkv [nimg * T, 3 W] bf16, D = W / heads;
 *     kernel 0 = the tcgen05 kernel (D = 64, 72 or 80) on at most max_ctas persistent CTAs (0: the encoder's grid), 1 = the mma.sync kernel (D = 80).
 *   novic_debug_siglip_map_attention: out [nimg, W] bf16 = the MAP head's attention of the fp32 query q [W] over kv [nimg * T, 2 W] bf16 (k | v).
 *   novic_debug_vit_layernorm: the encoder's LayerNorm kernel with every field of its parameters (W = 640, 768, 1024, 1152 or 1280): row r reads
 *     x + r * in_stride (first set to cls + pos0 when cls != NULL and r % cls_period == 0), y = LN(x; w1, b1) written back when store_x,
 *     out_bf [rows, W] = y, or LN(y; w2, b2) when w2 != NULL (out_bf may be NULL). */
int novic_debug_vit_gemm(const void* a, const void* w, int32_t M, int32_t N, int32_t K, int32_t epi, int32_t act, int32_t direct, const float* bias,
                         void* dst, int32_t ld, const float* table, int32_t patches, int32_t tok0, int32_t path, int32_t grid_div, void* stream);
int novic_debug_vit_attention(const void* qkv, int32_t nimg, int32_t T, int32_t W, int32_t heads, int32_t kernel, int32_t max_ctas, void* out, void* stream);
int novic_debug_siglip_map_attention(const void* kv, const float* q, int32_t nimg, int32_t T, int32_t W, int32_t heads, void* out, void* stream);
int novic_debug_vit_layernorm(float* x, int64_t in_stride, const float* w1, const float* b1, const float* w2, const float* b2, int32_t store_x, void* out_bf,
                              int32_t rows, int32_t W, float eps, const float* cls, const float* pos0, int32_t cls_period, void* stream);

/* Per-kernel-class device timing for roofline reports.  novic_kernel_timing(1) makes every subsequent direct
 * (non-graph) launch record a CUDA-event pair on its stream; novic_kernel_times() synchronises and returns the
 * accumulated milliseconds and launch counts per class, then clears.  Classes, in order: embed-prep, prefix GEMM,
 * QKV GEMM, attention, out-proj GEMM, FFN1 GEMM, FFN2 GEMM (also the fused out-proj + feed-forward block kernel), logits GEMM,
 * selection, other (n_classes >= 10). */
int novic_kernel_timing(int32_t enable);
int novic_kernel_times(double* ms_out, int64_t* count_out, int32_t n_classes);

/* Measurement aid (bench.py's in-graph roofline numbers, tools/ablate.py): keep_mask = bit set of kernel classes (bit k = class k
 * in the order above) whose launches are issued; the launches of all other classes are dropped, so a captured decode then
 * consists of that class's launches back to back, with their real arguments.  Results are meaningless while a mask is set.
 * keep_mask = 0 restores normal operation.  Drops the handle's cached graphs. */
int novic_debug_keep_classes(NovicHandle* h, uint32_t keep_mask);

/* Tuning aid: enable = 1 + n arms CTA (0,1) of the n-th GEMM launch from now to record clock64() at numbered phase
 * points; a later call returns the 32 recorded slots (out16: room for 32 int64, may be NULL) and re-arms / disarms (enable = 0). */
int novic_debug_trace(int64_t* out16, int32_t enable);

/* Byte offset of a named workspace buffer (ein, ebf, x, xn, xfin, q, ao, hb, kv, part) for the same arguments as
 * novic_workspace_bytes; lets tests inspect intermediates. */
int novic_debug_ws_offset(const NovicHandle* h, int64_t num_embeds, int32_t seqs_per_embed, int32_t rows_per_seq,
                          const char* name, size_t* offset_out);

/* The test-suite's own memory checker (compute-sanitizer is not available on the target pool).  novic_debug_redzone(bytes) makes every
 * buffer that the library carves out of a caller-owned workspace (novic_workspace_bytes / novic_train_workspace_bytes / weight buffers;
 * call it before those) be followed by `bytes` (a multiple of 256) that no kernel may touch; 0 restores the packed layout.
 * novic_debug_zones lists the untouchable (offset, length) ranges - guard bands plus alignment gaps - of a workspace: kind 0 = the
 * decode / teacher-forced workspace for the arguments of novic_workspace_bytes, kind 1 = the training workspace for the arguments
 * (B, M, C) of novic_train_workspace_bytes.  Returns the number of ranges (pairs_out: room for `cap` pairs, may be NULL) or -1. */
int novic_debug_redzone(size_t bytes);
int64_t novic_debug_zones(const NovicHandle* h, int32_t kind, int64_t num_embeds, int32_t seqs_per_embed, int32_t rows_or_cols,
                          uint64_t* pairs_out, int64_t cap);

/* Kernel launches issued by this process through the library since load (bench.py's gpu_launches). */
int64_t novic_launch_count(void);
/* Device-side watchdog word (non-zero after a kernel trapped on a stuck mbarrier). */
int novic_watchdog(uint32_t* code_out);
/* 0/1: capture decode loops into CUDA graphs (default 1). */
int novic_set_use_graphs(NovicHandle* h, int32_t enable);

#ifdef __cplusplus
}
#endif
#endif /* NOVIC_B200_H_ */
