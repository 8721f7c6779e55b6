/* vdk_b200.h — C ABI of libvdk_b200.so, the sm_100a implementation of DORAEMON's (wuji3/visiondk)
 * embedding hot path.  The reference is pure Python and has no FFI of its own (SURVEY.md §8b); each
 * entry point below names the reference call site (file:line under /root/reference) whose arithmetic
 * it replaces.  A maintainer binds these with ctypes (INTEGRATION.md shows the stubs).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller unless the name says `host`;
 *   - `stream` is a cudaStream_t passed as void*; calls enqueue work and return without synchronising;
 *   - nothing is allocated behind the caller: scratch comes in as `workspace` (+ a *_workspace_bytes query);
 *   - return value: VDK_OK (0) or a negative VDK_ERR_*; vdk_last_error_string() explains the last failure
 *     on the calling thread.  There is no CPU fallback: without a CUDA device every compute call fails.
 */
#ifndef VDK_B200_H_
#define VDK_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VDK_OK 0
#define VDK_ERR_INVALID (-1)   /* bad argument / unsupported shape */
#define VDK_ERR_CUDA (-2)      /* a CUDA runtime or driver call failed */
#define VDK_ERR_WORKSPACE (-3) /* workspace too small */
#define VDK_ERR_OVERFLOW (-4)  /* a candidate buffer overflowed; caller must take the wide path */

/* ---- library ------------------------------------------------------------------------------- */
int vdk_version(void);                    /* major*10000 + minor*100 + patch */
const char* vdk_last_error_string(void);  /* thread-local, never NULL */
/* 0 when a device of compute capability 10.x is present and usable, else VDK_ERR_CUDA. */
int vdk_device_check(void);

/* ---- dense contraction: D = epilogue(A . B^T) ---------------------------------------------- */
/* Replaces the cuBLAS/cuDNN GEMMs inside timm's ConvNeXt/ViT blocks that models/faceX/backbone/
 * timm_wrapper.py:52 runs (pointwise Linear layers, patchify convs as GEMMs) and the neck Linear
 * (timm_wrapper.py:36).  A is [M,K] row-major (pitch lda), B is [N,K] row-major (pitch ldb) — the
 * layout of nn.Linear.weight — both 16-bit (bf16 or fp16); accumulation is fp32 on tcgen05/TMEM. */
#define VDK_DTYPE_BF16 0
#define VDK_DTYPE_FP16 1
#define VDK_DTYPE_FP32 2

#define VDK_EPI_NONE 0           /* D = acc (+ bias[n]) */
#define VDK_EPI_GELU 1           /* D = gelu(acc + bias[n]): nn.GELU()'s erf form evaluated as 0.5 x (1 + tanh(x (c1 + c3 x^2))) with
                                    (c1, c3) fitted to it (max deviation 3.1e-4) in fp16x2; |err| <= 6e-4 |x| (tests/test_gemm_gpu.py) */
#define VDK_EPI_SCALE_RESIDUAL 2 /* D = residual[m,n] + gamma[n] * (acc + bias[n])  (ConvNeXt layer-scale; gamma = 1: plain residual) */
#define VDK_EPI_LAYERNORM 3      /* D = LayerNorm_N(acc + bias) * gamma + beta; the tile must span the row (N <= 256) */
#define VDK_EPI_MUL_GELU_GRAD 4  /* D = acc * gelu'(residual[m,n]): dgrad through the MLP's GELU (residual = saved pre-activation) */
/* Kernel variants are chosen per shape (CTA pairs for long-K GEMMs, a pipelined auxiliary-tile epilogue for GELU' / saved
 * pre-activations); the tuning switches VDK_GEMM_PAIR / VDK_GEMM_AUXPIPE (environment, read once) force them for tests. */

typedef struct vdk_gemm_desc {
  const void* A; /* [M,K] 16-bit, pitch lda */
  const void* B; /* [N,K] 16-bit, pitch ldb (nn.Linear.weight layout) */
  void* D;       /* [M,N] out_dtype, pitch ldd */
  int M, N, K, lda, ldb, ldd;
  int in_dtype, out_dtype, epilogue;
  const float* bias;    /* [N] or NULL */
  const float* gamma;   /* [N]: layer-scale (SCALE_RESIDUAL) or LayerNorm weight (LAYERNORM) */
  const float* beta;    /* [N]: LayerNorm bias */
  const void* residual; /* [M,ldr], dtype of D (SCALE_RESIDUAL) */
  int ldr;
  float ln_eps;
  int split_k; /* > 1: K is split over split_k CTAs per tile whose fp32 partials are atomically added into a
                  ZEROED fp32 D (skinny-M neck GEMM, timm_wrapper.py:36); epilogue NONE, no bias */
  long long split_stride; /* split_k > 1 only.  0: partials are atomically added into a zeroed D.  > 0 (elements):
                             split s stores its partial into the slab D + s*split_stride; the effective number of
                             splits is min(split_k, ceil(K/64)) rounded so that every split is non-empty — query it
                             with vdk_gemm_effective_splits.  Deterministic. */
  void* aux_out;  /* VDK_EPI_GELU only, may be NULL: also store the pre-activation acc + bias [M,ldd] (saved for backward) */
  int trans_a; /* 1: A is stored [K,M] row-major (pitch lda >= M): the contraction index is the slow dimension */
  int trans_b; /* 1: B is stored [K,N] row-major (pitch ldb >= N).  Backward GEMMs use these: dgrad
                  dX = dY . W (B = W stored [N_out,K_in] = [K,N] of this contraction) and wgrad dW = dY^T . X
                  (both operands stored with the token index slow) need no transposed copies. */
} vdk_gemm_desc;
int vdk_gemm(const vdk_gemm_desc* desc, void* stream);
/* Number of K splits vdk_gemm will actually use for (K, split_k). */
int vdk_gemm_effective_splits(int K, int split_k);

/* Positional convenience form of vdk_gemm (split_k = 1, no LayerNorm). */
int vdk_gemm_tn(const void* A, const void* B, void* D, int M, int N, int K, int lda, int ldb, int ldd,
                int in_dtype,          /* VDK_DTYPE_BF16 | VDK_DTYPE_FP16 */
                int out_dtype,         /* VDK_DTYPE_BF16 | VDK_DTYPE_FP16 | VDK_DTYPE_FP32 */
                int epilogue,          /* VDK_EPI_* */
                const float* bias,     /* [N] or NULL */
                const float* gamma,    /* [N], VDK_EPI_SCALE_RESIDUAL only */
                const void* residual,  /* [M,ldr] same dtype as D, VDK_EPI_SCALE_RESIDUAL only */
                int ldr, void* stream);

/* ---- ConvNeXt embedding forward (eval) ------------------------------------------------------ */
/* Replaces TimmWrapper.forward (models/faceX/backbone/timm_wrapper.py:51-54: timm ConvNeXt features with
 * num_classes=0, global_pool='' -> BatchNorm2d -> Flatten -> Linear -> BatchNorm1d, :30-38) followed by
 * F.normalize (models/faceX/face_model.py:139).  All pointers are device pointers to weights the caller packed
 * (visiondk_b200/backbone.py: layouts below); activations are NHWC bf16 in `workspace`. */
#define VDK_CONVNEXT_MAX_BLOCKS 64

typedef struct vdk_convnext_block {
  const float* dw_w;  /* depthwise 7x7 taps, [49][C] fp32 (tap-major, channel contiguous) */
  const float* dw_b;  /* [C] */
  const float* ln_w;  /* [C] LayerNorm(eps 1e-6) */
  const float* ln_b;  /* [C] */
  const void* fc1_w;  /* [4C, C] bf16 (nn.Linear.weight) */
  const float* fc1_b; /* [4C] */
  const void* fc2_w;  /* [C, 4C] bf16 */
  const float* fc2_b; /* [C] */
  const float* gamma; /* [C] layer scale */
  /* training only (may be NULL for inference): */
  const float* dw_w_flip; /* [49][C] taps in reverse order (backward-data of the depthwise conv) */
  const void* fc2_wg;     /* [C, 4C] bf16: gamma[c] * fc2.weight[c, :] (dgrad through layer scale) */
} vdk_convnext_block;

typedef struct vdk_convnext_down {
  const float* ln_w;   /* [Cin] LayerNorm2d(eps 1e-6) */
  const float* ln_b;   /* [Cin] */
  const void* conv_w;  /* [Cout, 4*Cin] bf16, K order (kh, kw, cin) */
  const float* conv_b; /* [Cout] */
} vdk_convnext_down;

typedef struct vdk_convnext_net {
  int image_size; /* square input side, multiple of 32 */
  int feat_dim;   /* embedding width (neck Linear out_features) */
  int depths[4];
  int dims[4];
  const void* stem_w;     /* [dims[0], 48] bf16, K order (c, kh, kw) = Conv2d(3,C0,4,4).weight flattened */
  const float* stem_b;    /* [dims[0]] */
  const float* stem_ln_w; /* [dims[0]] */
  const float* stem_ln_b;
  vdk_convnext_down down[4]; /* down[0] unused */
  vdk_convnext_block blocks[VDK_CONVNEXT_MAX_BLOCKS]; /* stage-major */
  const float* head_ln_w; /* [dims[3]] model.head.norm */
  const float* head_ln_b;
  const void* neck_w;  /* [feat_dim, h*w*dims[3]] bf16, K order (h, w, c), BN2d/BN1d eval statistics folded in */
  const float* neck_b; /* [feat_dim] folded bias */
} vdk_convnext_net;

/* Building blocks of the forward, exported for unit parity tests (NHWC bf16 activations):
 *   vdk_dwconv7_ln        y = LayerNorm_C(depthwise7x7(x, pad 3) + bias)         timm ConvNeXtBlock.conv_dw + .norm
 *   vdk_layernorm_patchify out = LayerNorm_C(x), patch == 2: regrouped as 2x2/stride-2 patch rows [B*H/2*W/2, 4C]
 *                          in (kh, kw, c) order (timm downsample LayerNorm2d + the im2col of its Conv2d(k2,s2)) */
int vdk_dwconv7_ln(const void* x, int batch, int H, int W, int C, const float* w49, const float* bias,
                   const float* ln_w, const float* ln_b, float eps, void* y, void* stream);
int vdk_layernorm_patchify(const void* x, int batch, int H, int W, int C, const float* ln_w, const float* ln_b,
                           float eps, int patch, void* out, void* stream);

/* ---- ConvNeXt training forward / backward -------------------------------------------------- */
/* fp32 tensors in timm's own layouts (device pointers): the master parameters, or — same struct — their gradients.
 * Replaces the train-mode forward of TimmWrapper (timm_wrapper.py:51-54, BatchNorm batch statistics at :34,37) and
 * its autograd backward, i.e. `scaler.scale(loss).backward()` at engine/procedure/train.py:206. */
typedef struct vdk_convnext_block_tensors {
  float* dw_w;  /* conv_dw.weight [C,1,7,7] */
  float* dw_b;
  float* ln_w;  /* norm.weight */
  float* ln_b;
  float* fc1_w; /* mlp.fc1.weight [4C,C] */
  float* fc1_b;
  float* fc2_w; /* mlp.fc2.weight [C,4C] */
  float* fc2_b;
  float* gamma;
} vdk_convnext_block_tensors;
typedef struct vdk_convnext_down_tensors {
  float* ln_w;
  float* ln_b;
  float* conv_w; /* downsample.1.weight [Cout,Cin,2,2] */
  float* conv_b;
} vdk_convnext_down_tensors;
typedef struct vdk_convnext_tensors {
  float* stem_w; /* stem.0.weight [C0,3,4,4] */
  float* stem_b;
  float* stem_ln_w;
  float* stem_ln_b;
  vdk_convnext_down_tensors down[4];
  vdk_convnext_block_tensors blocks[VDK_CONVNEXT_MAX_BLOCKS];
  float* head_ln_w;
  float* head_ln_b;
  float* bn2_w; /* output_layer.0 (BatchNorm2d) */
  float* bn2_b;
  float* bn2_running_mean;
  float* bn2_running_var;
  float* lin_w; /* output_layer.2.weight [F, C3*h*w] in timm's (c,h,w) flatten order */
  float* lin_b;
  float* bn1_w; /* output_layer.3 (BatchNorm1d) */
  float* bn1_b;
  float* bn1_running_mean;
  float* bn1_running_var;
} vdk_convnext_tensors;

/* Refreshes the bf16 / permuted kernel-layout weights of `net` (whose pointer fields address caller-allocated
 * buffers) from the fp32 masters: stem_w, down[].conv_w, blocks[].{dw_w, fc1_w, fc2_w, fc2_wg}, neck_w (un-folded,
 * (h,w,c) order).  fp32 vectors (biases, norms, gamma) are used in place: point net's fields at the masters.
 * vdk_convnext_pack_flip then derives blocks[].dw_w_flip. */
int vdk_convnext_pack(const vdk_convnext_tensors* params, vdk_convnext_net* net, void* stream);
int vdk_convnext_pack_flip(const vdk_convnext_net* net, void* stream);
size_t vdk_convnext_train_workspace_bytes(const vdk_convnext_net* net, int batch);
/* images fp32 NCHW -> out_feats fp32 [batch, feat_dim] (NOT normalised: the head normalises).  Saves activations in
 * `workspace` for the backward; updates the BatchNorm running statistics in `params` with `bn_momentum`. */
int vdk_convnext_train_forward(const vdk_convnext_net* net, const vdk_convnext_tensors* params, const float* images,
                               int batch, float bn_momentum, float* out_feats, void* workspace, size_t workspace_bytes,
                               void* stream);
/* d_feats fp32 [batch, feat_dim] -> gradients ACCUMULATED (+=) into `grads` (same struct, timm layouts). */
int vdk_convnext_train_backward(const vdk_convnext_net* net, const vdk_convnext_tensors* params,
                                const vdk_convnext_tensors* grads, const float* d_feats, int batch, void* workspace,
                                size_t workspace_bytes, void* stream);
/* The same backward in consecutive UNIT ranges (unit 0 = neck + head LayerNorm, then per stage 3..0 one unit per block,
 * last block first, and one for the stage's downsample layer / the stem): lets the caller start the DDP all-reduce
 * (engine/vision_engine.py:509-510 wraps the model in DistributedDataParallel, whose buckets overlap the backward) of the
 * gradients a range completed while the next range computes.  Ranges must be issued in order and cover [0, units). */
int vdk_convnext_train_backward_units(const vdk_convnext_net* net);
int vdk_convnext_train_backward_range(const vdk_convnext_net* net, const vdk_convnext_tensors* params,
                                      const vdk_convnext_tensors* grads, const float* d_feats, int batch, void* workspace,
                                      size_t workspace_bytes, void* stream, int unit_begin, int unit_end);

/* Building blocks of the backward, exported for unit parity tests (NHWC bf16 activations, fp32 parameter grads +=):
 *   vdk_dwconv7             mode 0: LayerNorm_C(dwconv7(x)+bias) (rstd_out optional); mode 1: dwconv7(x) with `w49` (+addend)
 *                           — with reversed taps this is the depthwise backward-data pass
 *   vdk_dwconv7_wgrad       dw49[tap][c] += sum dconv * shifted x; dbias[c] += sum dconv
 *   vdk_layernorm_bwd       LayerNorm backward from the saved OUTPUT y and 1/sigma (patch = 2: through the 2x2 regrouping)
 *   vdk_batchnorm_train_*   BatchNorm over the rows of [rows, C] with batch statistics (running stats updated) */
int vdk_dwconv7(int mode, const void* x, int batch, int H, int W, int C, const float* w49, const float* bias,
                const float* ln_w, const float* ln_b, float eps, void* y, float* rstd_out, const void* addend, void* stream);
int vdk_dwconv7_wgrad(const void* x, const void* dconv, int batch, int H, int W, int C, float* dw49, float* dbias,
                      void* stream);
int vdk_layernorm_bwd(const void* dy, const void* y, const float* rstd, int batch, int H, int W, int C, const float* ln_w,
                      const float* ln_b, int patch, void* dx, const void* addend, float* dgamma, float* dbeta, void* stream);
int vdk_batchnorm_train_fwd(const void* x, int rows, int C, int is_bf16, const float* weight, const float* bias, float eps,
                            float momentum, void* y, float* save_mean, float* save_rstd, float* running_mean,
                            float* running_var, void* stream);
int vdk_batchnorm_train_bwd(const void* dy, const void* x, int rows, int C, int is_bf16, const float* weight,
                            const float* save_mean, const float* save_rstd, void* dx, float* dweight, float* dbias,
                            void* stream);

size_t vdk_convnext_workspace_bytes(const vdk_convnext_net* net, int batch);
/* images: fp32 NCHW [batch,3,S,S] (what the reference's DataLoader yields); embeddings: fp32 [batch, feat_dim],
 * L2-normalised when l2_normalize != 0 (extract_cbir semantics). */
int vdk_convnext_forward(const vdk_convnext_net* net, const float* images, int batch, int l2_normalize,
                         float* embeddings, void* workspace, size_t workspace_bytes, void* stream);

/* ---- ViT inference forward (Transformer backbones of the CBIR extract path) ------------------- */
/* Replaces the eval forward of TimmWrapper for `timm-vit_*` backbones (models/faceX/backbone/timm_wrapper.py:16-21,
 * 39-47, 51-54: timm VisionTransformer with num_classes=0, global_pool='' -> every token after the final LayerNorm,
 * then LayerNorm -> Flatten -> Linear -> BatchNorm1d) as run by FeatureExtractor.extract_cbir (face_model.py:120-144).
 * All 16-bit weights are bf16 in nn.Linear layout [out, in]; vectors fp32; everything device memory. */
#define VDK_VIT_MAX_BLOCKS 48
typedef struct vdk_vit_block {
  const float* ln1_w; const float* ln1_b;
  const void* qkv_w;  const float* qkv_b;   /* [3*dim, dim], [3*dim]: rows ordered (q | k | v) x head x 64 as in timm */
  const void* proj_w; const float* proj_b;  /* [dim, dim] */
  const float* ln2_w; const float* ln2_b;
  const void* fc1_w;  const float* fc1_b;   /* [4*dim, dim] */
  const void* fc2_w;  const float* fc2_b;   /* [dim, 4*dim] */
} vdk_vit_block;
typedef struct vdk_vit_net {
  int image_size, patch, dim, depth, heads, feat_dim;
  const void* patch_w;      /* [dim, Kp] bf16, Kp = 3*patch*patch rounded up to 8, (c, kh, kw) order, zero padded */
  const float* patch_b;     /* [dim] */
  const float* cls_token;   /* [dim] */
  const float* pos_embed;   /* [1 + (image_size/patch)^2, dim] */
  const float* ones;        /* [dim] of 1.0f (layer-scale slot of the residual epilogue: timm's default ViT has none) */
  vdk_vit_block blocks[VDK_VIT_MAX_BLOCKS];
  const float* norm_w; const float* norm_b;        /* model.norm, eps 1e-6 */
  const float* neck_ln_w; const float* neck_ln_b;  /* output_layer.0, eps 1e-5 */
  const void* neck_w;       /* [feat_dim, tokens*dim] bf16 with BatchNorm1d (eval) folded in */
  const float* neck_b;      /* [feat_dim] folded */
  /* timm's `pre_norm=True` variants (vit_*_clip_*: CLIP towers): a LayerNorm right after cls / position (model.norm_pre),
   * a bias-free patch embedding (patch_b == NULL) and LayerNorm eps 1e-5.  NULL / 0 = the plain ViT above (eps 1e-6).
   * Inference only: vdk_vit_train_* refuse a net with norm_pre_w set. */
  const float* norm_pre_w; const float* norm_pre_b;
  float ln_eps;             /* eps of norm_pre, the block norms and model.norm; 0 selects 1e-6 */
} vdk_vit_net;
size_t vdk_vit_workspace_bytes(const vdk_vit_net* net, int batch);
/* images: fp32 NCHW [batch,3,S,S]; embeddings: fp32 [batch, feat_dim], L2-normalised when l2_normalize != 0. */
int vdk_vit_forward(const vdk_vit_net* net, const float* images, int batch, int l2_normalize, float* embeddings,
                    void* workspace, size_t workspace_bytes, void* stream);
/* softmax(Q K^T / sqrt(d)) V on the qkv Linear's output as stored: qkv bf16 [batch, tokens, 3, heads, 64] ->
 * out bf16 [batch, tokens, heads*64]  (timm Attention.forward, scores never written to memory). */
int vdk_attention_fwd(const void* qkv, int batch, int tokens, int heads, int head_dim, void* out, void* stream);

/* ---- ViT training forward / backward (BASELINE config 3: ViT-B/16 + CircleLoss) ----------------------------------- */
/* fp32 tensors in timm layouts (parameters, or their gradients): what TimmWrapper('vit_*').train() holds. */
typedef struct vdk_vit_block_tensors {
  float* ln1_w; float* ln1_b; float* qkv_w; float* qkv_b; float* proj_w; float* proj_b;
  float* ln2_w; float* ln2_b; float* fc1_w; float* fc1_b; float* fc2_w; float* fc2_b;
} vdk_vit_block_tensors;
typedef struct vdk_vit_tensors {
  float* patch_w;   /* [dim, 3, P, P] */
  float* patch_b; float* cls_token; float* pos_embed;
  vdk_vit_block_tensors blocks[VDK_VIT_MAX_BLOCKS];
  float* norm_w; float* norm_b; float* neck_ln_w; float* neck_ln_b;
  float* lin_w;     /* output_layer.2.weight [feat_dim, tokens*dim] */
  float* lin_b;
  float* bn1_w; float* bn1_b; float* bn1_running_mean; float* bn1_running_var;  /* output_layer.3 */
} vdk_vit_tensors;
/* fp32 masters -> the bf16 GEMM weights of `net` (patch_w, qkv/proj/fc1/fc2, neck_w UNfolded: BatchNorm1d runs on batch
 * statistics in train mode).  Vector pointers of `net` are set by the caller (they may alias the masters). */
int vdk_vit_pack(const vdk_vit_tensors* params, vdk_vit_net* net, void* stream);
size_t vdk_vit_train_workspace_bytes(const vdk_vit_net* net, int batch);
/* Train-mode forward of TimmWrapper('vit_*') (timm_wrapper.py:51-54; neck :42-47 with BatchNorm1d batch statistics,
 * running stats updated): images fp32 NCHW -> out_feats fp32 [batch, feat_dim]; activations saved in `workspace`.
 * Needs 3*patch*patch % 8 == 0; any token count (the attention backward runs the mma.sync kernel up to 208 tokens, the tcgen05
 * pair of vdk_attention_bwd_tc beyond). */
int vdk_vit_train_forward(const vdk_vit_net* net, const vdk_vit_tensors* params, const float* images, int batch, float bn_momentum,
                          float* out_feats, void* workspace, size_t workspace_bytes, void* stream);
/* d_feats fp32 [batch, feat_dim] -> gradients ACCUMULATED (+=) into `grads`. */
int vdk_vit_train_backward(const vdk_vit_net* net, const vdk_vit_tensors* params, const vdk_vit_tensors* grads, const float* d_feats,
                           int batch, void* workspace, size_t workspace_bytes, void* stream);
/* The same backward in consecutive unit ranges (0 = neck + final LayerNorm, 1..depth = blocks depth-1..0, depth+1 = cls / position /
 * patch embedding): the DDP overlap of vdk_convnext_train_backward_range for Transformer backbones. */
int vdk_vit_train_backward_units(const vdk_vit_net* net);
int vdk_vit_train_backward_range(const vdk_vit_net* net, const vdk_vit_tensors* params, const vdk_vit_tensors* grads,
                                 const float* d_feats, int batch, void* workspace, size_t workspace_bytes, void* stream, int unit_begin,
                                 int unit_end);
/* unit-test surface of the attention pair: forward that also saves the log2-domain log-sum-exp [batch, heads, tokens], and
 * the backward dqkv = d(attention)/d(qkv) for d_out (both [batch, tokens, heads*64] bf16). */
int vdk_attention_fwd_lse(const void* qkv, int batch, int tokens, int heads, int head_dim, void* out, float* lse2, void* stream);
int vdk_attention_bwd(const void* qkv, const void* out, const void* d_out, const float* lse2, int batch, int tokens, int heads,
                      int head_dim, void* dqkv, void* stream);
/* The same backward on tcgen05 for any token count (the mma.sync kernel above keeps one head's P in shared memory and stops at
 * 208 tokens).  Replaces timm's Attention backward inside `scaler.scale(loss).backward()` (engine/procedure/train.py:206) for long
 * sequences (ViT-B/8 at 224^2: 785 tokens, ViT-B/16 at 384^2: 577).  Two kernels on `stream`; no atomics, so dqkv is the same bits on every run.
 * workspace: caller-owned device memory of at least vdk_attention_bwd_tc_workspace_bytes(...) bytes, 16-byte aligned (holds
 * D = rowsum(d_out * out) per (image, head, token)).  head_dim must be 64.  Host-only sizing: returns 0 for a bad shape. */
size_t vdk_attention_bwd_tc_workspace_bytes(int batch, int tokens, int heads, int head_dim);
int vdk_attention_bwd_tc(const void* qkv, const void* out, const void* d_out, const float* lse2, int batch, int tokens, int heads,
                         int head_dim, void* dqkv, void* workspace, size_t workspace_bytes, void* stream);

/* ---- margin-softmax heads + cross-entropy --------------------------------------------------- */
/* Replaces ArcFace.forward (models/faceX/head/arcface.py:20-36), CircleLoss.forward (models/faceX/head/
 * circleloss.py:21-43), nn.CrossEntropyLoss(label_smoothing) (models/losses/loss.py:71-73) and their autograd
 * backward, as called at engine/procedure/train.py:196.  fp32 in / fp32 out like the reference (no autocast on the
 * face path); the three contractions run on tcgen05 with a 3-way bf16 operand split (fp32-grade accuracy). */
#define VDK_HEAD_ARCFACE 0
#define VDK_HEAD_CIRCLELOSS 1
#define VDK_HEAD_MV_SOFTMAX 2 /* MV_Softmax.forward, models/faceX/head/mv_softmax.py:25-44 */

typedef struct vdk_head_desc {
  int kind;                 /* VDK_HEAD_* */
  int batch, feat_dim, num_class;
  float margin_arc, margin_am, scale; /* ArcFace(margin_arc, margin_am, scale); scale also MV_Softmax */
  float margin, gamma;                /* CircleLoss(margin, gamma); margin also MV_Softmax */
  float label_smooth;                 /* CrossEntropyLoss(label_smoothing) */
  float mv_weight;                    /* MV_Softmax(is_am, margin, mv_weight, scale) */
  int is_am;
} vdk_head_desc;

size_t vdk_head_workspace_bytes(const vdk_head_desc* d);
/* feats fp32 [B,D]; weight fp32 [D,C] (the head Parameter); labels int64 [B].
 * logits: fp32 [B,C] or NULL; loss: device scalar (mean CE); row_lse: fp32 [B] saved for the backward;
 * cos_saved: fp32 [B,C] clamped cos(theta) or NULL. */
int vdk_head_forward(const vdk_head_desc* d, const float* feats, const float* weight, const int64_t* labels,
                     float* logits, float* loss, float* row_lse, float* cos_saved, void* workspace,
                     size_t workspace_bytes, void* stream);
/* Fused backward of mean-CE(head(feats)) (dlogits == NULL; grad_loss: device scalar or NULL for 1), or the head-only
 * backward for a caller-supplied dlogits fp32 [B,C] (row_lse / grad_loss ignored).  dfeats [B,D], dweight [D,C]. */
int vdk_head_backward(const vdk_head_desc* d, const float* feats, const float* weight, const int64_t* labels,
                      const float* row_lse, const float* grad_loss, const float* dlogits, float* dfeats,
                      float* dweight, void* workspace, size_t workspace_bytes, void* stream);

/* ---- optimizer step -------------------------------------------------------------------------- */
/* Replaces Trainer.update's clip_grad_norm_(max_norm=10) -> SGD step -> zero_grad -> ModelEMA.update
 * (engine/procedure/train.py:203-215, engine/optimizer.py:119-121, models/ema.py:28-37) on FLAT fp32 buffers
 * (parameters, gradients, momentum and EMA of one param group laid out contiguously by the caller). */
size_t vdk_grad_sumsq_workspace_bytes(void);
/* total_sumsq (device double) = [accumulate ? previous : 0] + sum(grads^2); deterministic summation order. */
int vdk_grad_sumsq(const float* grads, int64_t n, double* total_sumsq, int accumulate, void* workspace,
                   size_t workspace_bytes, void* stream);
/* One param group: g *= min(1, max_norm / (sqrt(total_sumsq) + 1e-6)); g += wd * p; buf = first_step ? g : mom*buf + g;
 * p -= lr * buf; ema = ema*d + (1-d)*p (ema may be NULL); g = 0 if zero_grad. */
int vdk_sgd_clip_ema_step(float* params, float* grads, float* momentum_buf, float* ema, int64_t n,
                          const double* total_sumsq, float max_norm, float lr, float momentum, float weight_decay,
                          int first_step, float ema_decay, float ema_one_minus_decay, int zero_grad, void* stream);
/* EMA of non-parameter float state (BatchNorm running statistics): ema = ema*d + (1-d)*src. */
int vdk_ema_update(float* ema, const float* src, int64_t n, float decay, float one_minus_decay, void* stream);

/* ---- retrieval: L2-normalise -> inner product -> top-k -------------------------------------- */
/* Replaces F.normalize at models/faceX/face_model.py:139, faiss index.add at
 * engine/cbir/evaluation.py:166-168 and faiss index.search at engine/cbir/evaluation.py:193
 * (cbir_eval.py:95,116).  Semantics: exact inner-product top-k; scores are the canonical fp32 scores
 * defined in oracle/retrieval.py (fixed-order fp64 accumulation), order = (score desc, id asc),
 * ids are int64, missing entries are id -1 / score -inf like faiss. */

/* Row preparation.  x: fp32 [n, dim] (pitch dim).  If `normalize`: xn = x / max(||x||, 1e-12) (F.normalize),
 * else xn = x.  Writes xn (fp32), xh = fp16(xn), row_norm[n] = ||xn||, row_err[n] >= ||xn - xh||.
 * Any of xn / row_norm may alias NULL to skip that output; xn may alias x (in place). */
int vdk_rows_prepare(const float* x, int64_t n, int dim, int normalize, float* xn, void* xh, float* row_norm,
                     float* row_err, void* stream);

typedef struct vdk_topk_plan {
  int64_t n_query;       /* rows of the query block */
  int64_t n_gallery;     /* rows of the (local shard of the) gallery */
  int dim;               /* embedding width, multiple of 64, <= 512 */
  int k;                 /* neighbours wanted, 1..1024 */
  int cand_capacity;     /* per-query slots for one range's admitted candidates (multiple of 32, >= 2k) */
  int carry_capacity;    /* per-query slots for survivors carried between ranges (in [2k, 4096]) */
  int n_stages;          /* gallery is scanned in n_stages ranges; thresholds tighten between them */
  int dense_mask;        /* bit s set: range s is scored densely (no admission threshold; must fit cand_capacity);
                            bit 0 is implied.  An all-dense plan cannot overflow a segment (the wide path). */
  int64_t stage_end[8];  /* exclusive end row of each stage (last == n_gallery) */
} vdk_topk_plan;

/* Fills stage boundaries / capacity for the given problem; returns VDK_OK. */
int vdk_topk_plan_default(vdk_topk_plan* plan, int64_t n_query, int64_t n_gallery, int dim, int k);
/* Scratch bytes vdk_ip_topk needs for this plan. */
size_t vdk_topk_workspace_bytes(const vdk_topk_plan* plan);

/* Exact inner-product top-k of q against g.
 *   q32/g32  : fp32 rows (what the scores are defined on), qh/gh: their fp16 copies from vdk_rows_prepare
 *   q_norm/q_err : per-query ||q|| and fp16 rounding-error norm; g_norm_max/g_err_max: device scalars, the
 *                  maxima over the gallery (vdk_reduce_max) — they bound the tensor-core score error.
 *   id_offset : added to every returned id (shard offset under multi-GPU sharding).
 *   out_scores: fp32 [n_query,k], out_ids: int64 [n_query,k].
 *   status    : device int32[4]: {overflow_rows, max_candidates_seen, rerank_rows_max, reserved}. */
int vdk_ip_topk(const vdk_topk_plan* plan, const float* q32, const void* qh, const float* q_norm,
                const float* q_err, const float* g32, const void* gh, const float* g_norm_max,
                const float* g_err_max, int64_t id_offset, float* out_scores, int64_t* out_ids, int32_t* status,
                void* workspace, size_t workspace_bytes, void* stream);

/* The two halves of vdk_ip_topk, for the SHARDED search (gallery rows split over GPUs, BASELINE config 4):
 *   vdk_ip_topk_filter  scans this shard (thresholds, ranges, selects), leaves every query's candidates in `workspace` and
 *                       writes kth_lb_out[n_query]: a lower bound of the shard's k-th largest canonical score (-inf if the
 *                       shard holds fewer than k rows);
 *   -- the ranks turn what they publish into a lower bound T of the GLOBAL k-th canonical score: the element-wise max of
 *      kth_lb, or better vdk_ip_topk_rank_sketch + vdk_topk_bound_from_sketches below --
 *   vdk_ip_topk_rerank  re-scores canonically only the candidates that can still reach the global top-k
 *                       (approx >= kth_lb_global - eps) and emits this shard's list, padded with (-FLT_MAX, -1).
 * The merged result (vdk_topk_merge*) is bit-identical to the unsharded search.  kth_lb_global == NULL re-ranks everything
 * (what vdk_ip_topk does).  Same plan, workspace and stream for both calls. */
int vdk_ip_topk_filter(const vdk_topk_plan* plan, const void* qh, const float* q_norm, const float* q_err, const void* gh,
                       const float* g_norm_max, const float* g_err_max, float* kth_lb_out, int32_t* status, void* workspace,
                       size_t workspace_bytes, void* stream);
/* The scan stage by stage, for shards that exchange their bounds BETWEEN gallery ranges: runs stages [stage_begin, stage_end) of
 * the plan (stage_begin == 0 initialises the workspace).  ext_lb (device fp32 [n_query], nullable): a lower bound of the GLOBAL
 * k-th canonical score derived from what all shards published after the previous stage (vdk_topk_bound_from_sketches) — it
 * tightens this shard's admission threshold and carry list (a candidate below ext_lb - eps cannot reach the global top-k), so
 * that after every exchange each shard filters as if it had scanned the union of all shards' prefixes.  kth_lb_out as in
 * vdk_ip_topk_filter, never below ext_lb. */
int vdk_ip_topk_filter_stages(const vdk_topk_plan* plan, const void* qh, const float* q_norm, const float* q_err, const void* gh,
                              const float* g_norm_max, const float* g_err_max, int stage_begin, int stage_end, const float* ext_lb,
                              float* kth_lb_out, int32_t* status, void* workspace, size_t workspace_bytes, void* stream);
int vdk_ip_topk_rerank(const vdk_topk_plan* plan, const float* q32, const float* g32, int64_t id_offset,
                       const float* kth_lb_global, float* out_scores, int64_t* out_ids, void* workspace, size_t workspace_bytes,
                       void* stream);

/* What shards exchange between gallery ranges (sharded search; no counterpart in the reference, which replicates the index:
 * engine/cbir/evaluation.py:159-162).  After `stages_done` stages of the plan ran (vdk_ip_topk_filter_stages), writes
 * sketch_out[n_query][n_ranks]: for every query and every ranks[i] (host array, 1 <= ranks[i] <= k, at most 8) a lower bound of
 * the canonical score of this shard's ranks[i]-th best row so far (-inf if it holds fewer candidates).  ranks[i] == k reports the
 * select's own k-th bound. */
int vdk_ip_topk_rank_sketch(const vdk_topk_plan* plan, int stages_done, const int32_t* ranks, int n_ranks, float* sketch_out,
                            void* workspace, size_t workspace_bytes, void* stream);
/* sketches: device fp32 [n_shards][n_query][n_ranks] (the all-gathered sketch_out of every shard, disjoint rows).
 * bound_inout[q] = max(bound_inout[q], largest reported score t with sum over shards of max{ranks[i] : sketch[i] >= t} >= k):
 * a lower bound of the GLOBAL k-th canonical score — the `ext_lb` of the next vdk_ip_topk_filter_stages call and the
 * kth_lb_global of vdk_ip_topk_rerank. */
int vdk_topk_bound_from_sketches(const float* sketches, int n_shards, int64_t n_query, const int32_t* ranks, int n_ranks, int k,
                                 float* bound_inout, void* stream);

/* Device pointer (inside `workspace`) to int32[n_query] flags the last vdk_ip_topk set for rows whose candidate lists
 * overflowed; status[0] counts them.  Their results are incomplete and must be recomputed with an all-dense plan. */
int vdk_topk_row_flags(const vdk_topk_plan* plan, const void* workspace, size_t workspace_bytes,
                       const int32_t** row_flags);

/* Exhaustive exact top-k for a FEW queries: canonical scores against every gallery row, exact selection on
 * (score desc, id asc) keys.  No candidate capacity, so it cannot overflow: the last resort for queries flagged by
 * vdk_ip_topk even under an all-dense plan (thousands of exact duplicates of a top-k member) — faiss' flat search
 * (engine/cbir/evaluation.py:193) answers such queries, so this path must too.  q32: fp32 [n_query, dim] (already
 * normalised if the index is a cosine index).  workspace >= vdk_ip_topk_exhaustive_workspace_bytes(n_gallery). */
size_t vdk_ip_topk_exhaustive_workspace_bytes(int64_t n_gallery);
int vdk_ip_topk_exhaustive(const float* q32, int64_t n_query, const float* g32, int64_t n_gallery, int dim, int k,
                           int64_t id_offset, float* out_scores, int64_t* out_ids, void* workspace, size_t workspace_bytes,
                           void* stream);

/* Measurement hook: launches ONLY the score/filter kernel of vdk_ip_topk for gallery rows [lo, hi), reusing the
 * thresholds a previous vdk_ip_topk left in `workspace` (dense != 0: the threshold-free first-range variant).
 * bench.py brackets this call with CUDA events to time the dominant kernel in isolation. */
int vdk_score_range(const vdk_topk_plan* plan, const void* qh, const void* gh, int64_t lo, int64_t hi, int dense,
                    void* workspace, size_t workspace_bytes, void* stream);

/* Max over a float vector into a device scalar (gallery-wide error/norm bounds). */
int vdk_reduce_max(const float* x, int64_t n, float* out, void* stream);

/* Merge `n_lists` per-shard top-k lists (each [n_query,k], already ordered) into the global top-k with
 * the same (score desc, id asc) rule.  Replaces faiss' IndexShards merge (the reference uses replicas,
 * engine/cbir/evaluation.py:159-162; sharding is BASELINE config 4). */
int vdk_topk_merge(const float* scores, const int64_t* ids, int n_lists, int64_t n_query, int k, float* out_scores,
                   int64_t* out_ids, void* stream);

/* The exchange format of the sharded search: one 64-bit word per list entry, (fp32 score bits << 32) | uint32 id
 * (id -1, the padding, becomes 0xffffffff; global ids must therefore stay below 2^32 - 1), so that the ranks' lists travel in
 * ONE all-gather.  vdk_topk_pack: (scores, ids)[n] -> packed[n].  vdk_topk_merge_packed: packed [n_lists, n_query, k] ->
 * global top-k, same rule as vdk_topk_merge. */
int vdk_topk_pack(const float* scores, const int64_t* ids, int64_t n, void* packed, void* stream);
int vdk_topk_merge_packed(const void* packed, int n_lists, int64_t n_query, int k, float* out_scores, int64_t* out_ids,
                          void* stream);

/* Brute-force canonical scores for verification at full size: out[i] = canonical_score(q[qi[i]], g[gi[i]]). */
int vdk_ip_exact_pairs(const float* q32, const float* g32, int dim, const int64_t* qi, const int64_t* gi, int64_t n,
                       float* out, void* stream);

/* ---- eval-time image preprocessing (SURVEY.md §8f-3: the GPU input pipeline) ------------------------------------------ */
/* Replaces, for a BATCH of decoded RGB images of different sizes, the `val.augment` list of configs/faceX/{face,cbir}.yaml:
 * ResizeAndPadding2Square(size, training=False) (dataset/transforms.py:325-365: PIL Image.resize(BILINEAR) of the longer side
 * to `size`, centred on a black square), T.ToTensor (:466-468) and T.Normalize(mean, std) (:474-477).  Bit-exact with
 * Pillow's 8-bit resampling + torch's fp32 arithmetic (oracle/preprocess.py, pinned against the installed Pillow / torchvision).
 *   packed : DEVICE uint8, every image as [height][width][3] (RGB) at images[i].offset
 *   images : HOST array of n descriptors
 *   out    : DEVICE fp32 [n, 3, size, size]
 * The call computes the resampling coefficients on the host (double precision, like Pillow), uploads them and synchronises
 * the stream once before launching (JPEG decoding itself stays on the host: out of scope). */
typedef struct vdk_image_desc {
  int64_t offset;   /* bytes from `packed` to the image's first pixel */
  int width, height;
} vdk_image_desc;
size_t vdk_preprocess_workspace_bytes(const vdk_image_desc* images, int n, int size);
int vdk_preprocess_resize_pad_normalize(const uint8_t* packed, const vdk_image_desc* images, int n, int size, const float* mean,
                                        const float* std_, float* out, void* workspace, size_t workspace_bytes, void* stream);

/* Live kernel timing inside a real step (bench.py's roofline legs; not part of the reference's surface).  Between
 * vdk_prof_begin() and vdk_prof_end() every launch of the categories below is bracketed by two CUDA events on the stream it
 * is launched on; vdk_prof_end synchronises on them and returns, per category, the launch count, the summed event time and
 * the summed ALGORITHMIC flops / bytes of those launches.  Categories: 0 tcgen05 GEMM (vdk_gemm and every internal GEMM),
 * 1 depthwise 7x7 (forward+LN, data gradient, weight gradient), 2 attention (forward, backward), 3 retrieval score/filter,
 * 4 other.  Profiling perturbs the step (two event records per launch): never time a step with a profile open. */
typedef struct vdk_prof_total {
  long long launches;
  double ms;
  double flops;
  double bytes;
} vdk_prof_total;
#define VDK_PROF_CATEGORIES 5
int vdk_prof_begin(void);
int vdk_prof_end(vdk_prof_total* totals, int n_categories);

/* sizeof() of the by-pointer structs, in this order: vdk_gemm_desc, vdk_topk_plan, vdk_head_desc, vdk_convnext_net,
 * vdk_convnext_tensors, vdk_vit_net, vdk_vit_tensors.  Writes min(n, count) entries, returns the count: a binding checks its mirrors. */
int vdk_struct_sizes(size_t* out, int n);

#ifdef __cplusplus
}
#endif
#endif /* VDK_B200_H_ */
