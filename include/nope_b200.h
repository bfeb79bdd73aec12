/* nope_b200 -- C ABI of the B200-native NOPE inference hot path.
 *
 * The reference (nv-nguyen/nope) is pure Python/PyTorch and has no FFI of its own;
 * each entry point below names the reference function it replaces (paths relative to
 * the reference root).  All pointers are raw device pointers unless marked HOST; no
 * torch types cross this boundary.  Every function returns 0 on success and a negative
 * value on failure; nope_last_error() then returns a description (thread-local).
 * `stream` is a cudaStream_t passed as void* (NULL = default stream).
 *
 * Layout conventions at the boundary follow the reference's tensors:
 *   latent features   fp32 NCHW [B, C, 32, 32]           (encoder output, u_net input)
 *   poses             fp32 [B, N, 6]                     (6-D rotations, all_relativeR)
 *   embeddings        fp32 [B, N, C, 32, 32]             (pred_feat_templates)
 *   similarity        fp32 [B, N]; nearest_idx int64 [B, k]
 * Inside the library activations are NHWC fp16 and weights are repacked K-major fp16.
 *
 * ABI version 2 (round 2): nope_unet_set_option / get_option, caller-owned workspace
 * (nope_unet_workspace_bytes / nope_unet_set_workspace), nope_unet_profile_read reports executed and
 * algorithmic FLOPs, nope_op_conv_gn_fused, nope_topk_merge, nope_score_topk metric 2.
 */
#ifndef NOPE_B200_H
#define NOPE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct nope_unet nope_unet_t;

#define NOPE_METRIC_L2 0      /* reference "l2": -(sum_hw sqrt(sum_c (q-t)^4)), model.py:260-262 */
#define NOPE_METRIC_COSINE 1  /* extension: cosine of flattened descriptors (not in the reference) */
/* extension: occlusion-aware cosine -- the per-pixel cosine over channels (the encoder's
 * `sim_distance = nn.CosineSimilarity(dim=1)`, src/model/encoder/template.py:45) with similarities <=
 * threshold set to zero (`OcclusionAwareSimilarity`, src/model/encoder/base_template.py:67-75; threshold
 * 0.2 in configs/model/template_base.yaml), averaged over the 32x32 pixels */
#define NOPE_METRIC_COSINE_OCC 2

/* Thread-local message of the last failing call on this thread. */
const char* nope_last_error(void);

/* Library/ABI version and the SM architecture the kernels were built for ("sm_100a"). */
int nope_abi_version(void);
const char* nope_build_arch(void);

/* ---- engine lifetime ------------------------------------------------------------
 * Replaces construction of src/model/u_net/denoising_diffusion_pytorch/u_net.py:27-158
 * (UNet.__init__ with use_hard_up_down=True, dim_mults=(1,2,4,8), 8 groups,
 * pose_mlp_name="single_layer").  u_net_dim must be a multiple of 64; latent_ch <= 8;
 * latent_hw is the latent side (32 for 256x256 images). */
int nope_unet_create(nope_unet_t** out, int u_net_dim, int latent_ch, int latent_hw, int device);
void nope_unet_destroy(nope_unet_t* u);

/* Hand one tensor of the reference state_dict to the engine, by its reference key
 * (e.g. "downs.0.0.block1.proj.weight"; SURVEY.md 8b).  `data` is a HOST fp32 pointer,
 * contiguous, with `ndim` sizes in `shape`.  Unknown keys are rejected; encoder.* keys
 * are not accepted here (they go to nope_encoder_load_tensor below).
 * Replaces nn.Module.load_state_dict for the UNet; the shape-filtered partial load of
 * src/utils/weight.py:6-37 (skip keys whose shape does not match) is done by the Python mirror
 * (nope_b200.unet.load_checkpoint), this call rejects a mismatching shape. */
int nope_unet_load_tensor(nope_unet_t* u, const char* key, const float* data,
                          const int64_t* shape, int ndim);

/* Checks that every tensor was provided, repacks weights (OIHW fp32 -> K-major fp16,
 * pose projections concatenated into one GEMM) and uploads them. */
int nope_unet_finalize(nope_unet_t* u);

/* Tunables: hypotheses per chunk (workspace = ~5.5 MB per hypothesis), and the
 * convolution implementation: 0 = tcgen05 tensor cores, 128-pixel tiles, 1 = SIMT debug
 * twin, 2 = tcgen05 with CTA pairs (cta_group::2, 256-pixel tiles; default). */
int nope_unet_set_chunk(nope_unet_t* u, int hyps_per_chunk);
int nope_unet_set_conv_impl(nope_unet_t* u, int impl);
/* Named options:
 *   "precision" (before nope_unet_finalize): 0 = fp16 operands (default; embeddings ~1.3e-3 rel-L2 of the
 *       fp32 reference, u_net.py:160-198), 1 = exact weights: every weight is an fp16 pair W_hi + W_lo and
 *       each convolution accumulates A W_hi + A W_lo (2x the tensor-core work), 2 = split precision:
 *       exact weights and activations carried as fp16 pairs, A_hi W_hi + A_hi W_lo + A_lo W_hi (3x;
 *       the "parity" mode that meets the 1e-3 embedding tolerance with margin), 3 = bf16 operands and
 *       activations (BASELINE configs[2]; 8-bit mantissa: embeddings ~1e-2 of the fp32 reference),
 *       4 = split precision with single-fp16 tensors inside the ResnetBlocks (block2 convolutions run two
 *       products instead of three; embeddings ~5e-4: the fastest mode inside the 1e-3 tolerance);
 *   "fuse_gn" (default 1): GroupNorm + SiLU + pose bias + residual run in the epilogue of the producing
 *       convolution (Block.forward / ResnetBlock.forward, model_utils.py:237-279); 0 = separate
 *       gn_apply pass (round-1 schedule; also what conv_impl 0 / 1 use);
 *   "conv_impl": as nope_unet_set_conv_impl;
 *   "attn_impl": LinearAttention core, 0 = tcgen05 kernel at 32x32 / 16x16 (CUDA cores below 128 tokens),
 *       1 = CUDA-core kernel everywhere. */
int nope_unet_set_option(nope_unet_t* u, const char* name, int value);
int nope_unet_get_option(const nope_unet_t* u, const char* name, int* value);

/* Workspace ownership.  By default the engine owns one device slab and grows it on demand (a growth
 * synchronises the device and calls cudaMalloc).  A host framework that wants every byte to come from
 * its own allocator asks for the size and hands a buffer over; the sweep then never allocates and
 * fails if the buffer is too small.  hyps = min(chunk, B*N) hypotheses per chunk, refs = B,
 * scores = B*N (0 when no query is scored).  The buffer must stay alive while the engine uses it. */
int64_t nope_unet_workspace_bytes(nope_unet_t* u, int hyps, int refs, int scores);
int nope_unet_set_workspace(nope_unet_t* u, void* device_ptr, int64_t bytes, int hyps, int refs, int scores);

/* ---- the hot path -----------------------------------------------------------------
 * Sweep over the pose grid.  Replaces the Python loop of
 * PoseConditional.generate_templates (src/model/model.py:193-252) around
 * UNet.forward (u_net.py:160-198) and, when query_feat != NULL, the scoring and top-k of
 * PoseConditional.retrieval (model.py:254-266) fused onto the last layer.
 *   ref_feat   [B, C, hw, hw] fp32   encode_image(reference)
 *   poses      [B, N, 6] fp32        all_relativeR
 *   query_feat [B, C, hw, hw] fp32 or NULL
 *   out_emb    [B, N, C, hw, hw] fp32 or NULL (skip materialising the templates)
 *   out_sim    [B, N] fp32 or NULL   (requires query_feat)
 *   out_topv / out_topi  [B, k] fp32 / int64 or NULL; descending score, ties broken by
 *              the lowest index; indices are offset by idx_base (global index of this
 *              shard's first pose).  k = 0 skips the ranking.
 * Kernels are enqueued on `stream`; the call does not synchronise. */
int nope_unet_sweep(nope_unet_t* u, const float* ref_feat, const float* poses, int B, int N,
                    const float* query_feat, float* out_emb, float* out_sim, int k,
                    float* out_topv, int64_t* out_topi, int64_t idx_base, void* stream);

/* Similarity metric of the scoring fused onto the sweep's last layer (NOPE_METRIC_*; default l2, the only
 * one the reference implements, model.py:254-266).  occlusion_threshold is used by NOPE_METRIC_COSINE_OCC. */
int nope_unet_set_metric(nope_unet_t* u, int metric, float occlusion_threshold);

/* Number of kernels the last nope_unet_sweep call enqueued (for bench.py's gpu_launches). */
int64_t nope_unet_last_launch_count(const nope_unet_t* u);

/* Profiling hook for bench.py's roofline: when enabled, every tensor-core convolution
 * launch of subsequent sweeps is bracketed by CUDA events on the launching stream.
 * nope_unet_profile_read synchronises the device and returns the summed launch time
 * (ms), the summed EXECUTED FLOPs (2*M*N*K' per launch, K' counting the extra split-precision
 * K-segments), the summed ALGORITHMIC FLOPs (2*M*N*K of the layer, what the reference computes),
 * the launch count and the best single-launch executed TFLOP/s.  Enabling/disabling clears the
 * recorded events. */
int nope_unet_profile(nope_unet_t* u, int enable);
int nope_unet_profile_read(nope_unet_t* u, double* conv_ms, double* conv_flops, double* conv_alg_flops,
                           int64_t* conv_launches, double* max_launch_tflops);

/* ---- template encoder ----------------------------------------------------------------
 * FeatureExtractor.encode_image (src/model/encoder/template.py:47-53): ResNet-50 without
 * max-pool and with layer4 at stride 1 (src/model/encoder/resnet.py:93-152), eval-mode
 * BatchNorm folded into the convolutions, projector ReLU-1x1-ReLU-1x1, normalize=False.
 * Runs on the tcgen05 convolution kernel with split-precision (fp16 hi+lo) operands, so the
 * latents match the reference's fp32 path to 5e-5 rel-L2 (measured; tests assert 1.5e-4;
 * cuDNN TF32 / fp16 are 2-3e-3 off).  Keys are the reference's
 * `backbone.*` / `projector.*` names (HOST fp32 pointers, shape-checked); 256x256 inputs. */
typedef struct nope_encoder nope_encoder_t;
int nope_encoder_create(nope_encoder_t** out, int descriptor_size, int device);
void nope_encoder_destroy(nope_encoder_t* e);
int nope_encoder_load_tensor(nope_encoder_t* e, const char* key, const float* data,
                             const int64_t* shape, int ndim);
int nope_encoder_finalize(nope_encoder_t* e);
/* images [B, 3, 256, 256] fp32 NCHW (device) -> out [B, D, 32, 32] fp32 NCHW (device).
 * Any B >= 1: the engine walks the batch 32 images at a time (workspace ~80 MB per image of a chunk). */
int nope_encoder_encode(nope_encoder_t* e, const float* images, int B, float* out, void* stream);
int64_t nope_encoder_last_launch_count(const nope_encoder_t* e);

/* Score materialised templates against a query and rank them: the arithmetic of
 * PoseConditional.retrieval (model.py:254-266) after encode_image.
 *   query_feat [B, C, HW] fp32, emb [B, N, C, HW] fp32 -> sim [B, N], topv/topi [B, k]. */
int nope_score_topk(const float* query_feat, const float* emb, int B, int N, int C, int HW,
                    int metric, float occlusion_threshold, int k, float* out_sim, float* out_topv,
                    int64_t* out_topi, int64_t idx_base, void* stream);

/* Rank an existing similarity matrix sim [B, N] (used to merge per-GPU shards). */
int nope_topk(float* sim, int B, int N, int k, float* out_topv, int64_t* out_topi,
              int64_t idx_base, void* stream);

/* Multi-GPU merge (SURVEY.md 8e): each rank sweeps a contiguous slice of the pose grid and contributes
 * ONE packed record to a single all-gather:
 *   [ topv: B*k f32 | 1 pad float if B*k is odd | topi: B*k int64 (GLOBAL indices, -1 = padding) |
 *     similarity slice: B * n_local f32 (optional) | pad to a multiple of 4 floats ]
 * nope_topk_pack_floats gives the record length in floats (n_local_max = ceil(N / world)); records sit back to back
 * in the gathered buffer, so the length keeps every record's int64 block 8-byte aligned.
 * nope_topk_merge turns the `world` gathered records (each pack_floats long) into the global top-k
 * per batch row (descending, ties -> lowest index; identical on every rank) and, when has_sim, the
 * full similarity rows [B, N].  Rank r owns poses [r*per, min(N, (r+1)*per)). */
int64_t nope_topk_pack_floats(int B, int k, int n_local_max, int want_sim);
int nope_topk_merge(const float* gathered, int world, int64_t pack_floats, int B, int k, int N, int per,
                    int has_sim, float* out_sim, float* out_topv, int64_t* out_topi, void* stream);

/* ---- per-op entry points (parity tests drive single layers through these) -----------
 * All tensors fp32 NCHW device pointers; conversion to the internal NHWC fp16 layout
 * happens inside.  These calls synchronise the stream before returning.
 * conv: mode 0 = 3x3 pad 1 (model_utils.py:240), 1 = 1x1 (model_utils.py:269),
 *       2 = pixel-unshuffle(2)+1x1 (HardDownsample, model_utils.py:168-172; input is
 *       [n, C0, 2H, 2W], weight [Cout, 4*C0]), 3 = nearest-x2 upsample + 3x3 (HardUpsample,
 *       model_utils.py:161-165; input is [n, C0, H/2, W/2], weight [Cout, C0, 3, 3], folded
 *       inside into four 2x2 parity kernels).  x1 (optional) is concatenated after x0 along
 *       channels (u_net.py:186).  impl as in nope_unet_set_conv_impl. */
int nope_op_conv(int impl, int mode, const float* x0, int C0, const float* x1, int C1,
                 const float* weight, const float* bias, float* out, int n_img, int H, int W,
                 int Cout, void* stream);
/* Block.forward (model_utils.py:248-252): [SiLU](GroupNorm_G(conv(x) + bias)) with the
 * GroupNorm statistics taken from the convolution epilogue -- the fused path the sweep uses. */
int nope_op_conv_gn(int impl, int mode, const float* x0, int C0, const float* x1, int C1,
                    const float* weight, const float* bias, const float* gamma, const float* beta,
                    int G, int silu, float* out, int n_img, int H, int W, int Cout, void* stream);
/* The sweep's fused layer (conv_impl 2): out = [SiLU](GroupNorm_G(conv(x) + bias)) + chan_bias[n, c] +
 * residual[n / res_div] with everything after the convolution applied in its epilogue
 * (ResnetBlock.forward, model_utils.py:271-279; G = 0: no normalisation).  mode 0..2 as nope_op_conv.
 * precision as nope_unet_set_option.  chan_bias [n, Cout], residual [ceil(n / res_div), Cout, H, W]
 * (res_div 0: one residual image per input image), emit_out (optional) [n, 2] receives the sum and the
 * sum of squares of the stored output (the GroupNorm(1) statistics handed to a following pre-norm). */
int nope_op_conv_gn_fused(int mode, int precision, const float* x0, int C0, const float* x1, int C1,
                          const float* weight, const float* bias, const float* gamma, const float* beta,
                          int G, int silu, const float* chan_bias, const float* residual, int res_div,
                          float* out, float* emit_out, int n_img, int H, int W, int Cout, void* stream);
/* y = [SiLU](GroupNorm_G(x)) + chan_bias[n, c] + residual   (model_utils.py:237-253,271-279) */
int nope_op_groupnorm(const float* x, const float* gamma, const float* beta, int G, int silu,
                      const float* chan_bias, const float* residual, float* out, int n_img,
                      int C, int H, int W, void* stream);
/* LinearAttention core on qkv [n, 384, H, W] -> [n, 128, H, W] (model_utils.py:403-417).
 * impl 0: tcgen05 kernel (both contractions on tensor cores, H*W a multiple of 128), 1: CUDA cores. */
int nope_op_linear_attention(int impl, const float* qkv, float* out, int n_img, int H, int W, void* stream);
/* Attention core on qkv [n, 384, H, W] -> [n, 128, H, W], H*W <= 32 (model_utils.py:376-388) */
int nope_op_attention(const float* qkv, float* out, int n_img, int H, int W, void* stream);
/* nearest x2 upsample (model_utils.py:161-163) */
int nope_op_upsample2x(const float* x, float* out, int n_img, int C, int H, int W, void* stream);

/* Debug: run the sweep for B=1 and copy the activation named `tap` (oracle tap names,
 * e.g. "downs.0.0", "mid.1", "ups.2.3", "final_conv.0") to out as fp32 NCHW [N, C, H, W]. */
int nope_unet_debug_tap(nope_unet_t* u, const float* ref_feat, const float* poses, int N,
                        const char* tap, float* out, int64_t out_capacity_floats,
                        int* out_C, int* out_H, void* stream);

/* ---- LDM variant (SURVEY.md 8 f2) ------------------------------------------------------
 * UNetModelPose (src/model/u_net/ldm/adapt_openaimodel.py:14-158 over ldm/openaimodel.py:428-760
 * and ldm/attention.py:149-277; configs/model/vae_cin_ldm.yaml): ResBlocks + SpatialTransformers
 * (self-attention on tcgen05, the one-token pose cross-attention folded to a per-hypothesis
 * channel vector, GEGLU feed-forward), strided-conv down / nearest-x2+conv up, emb = 0.
 * Supported configuration: channel_mult (1, 2, 4), 2 ResBlocks per level, attention at every
 * level, num_head_channels 32, transformer_depth 1, injecting_condition_twice false,
 * pose_mlp "single_layer", model_channels a multiple of 256, 32x32 latents.
 * Keys are the reference's state_dict names (628 tensors for model_channels 256; the unused
 * time_embed.* entries are accepted); HOST fp32 pointers, shape-checked.  The VAE encoder
 * (diffusers AutoencoderKL, not part of the reference tree) is out of scope: the sweep takes
 * latents.  Arguments of nope_ldm_sweep are those of nope_unet_sweep with
 * ref_feat / query_feat = [B, latent_ch, 32, 32] latents. */
typedef struct nope_ldm nope_ldm_t;
int nope_ldm_create(nope_ldm_t** out, int model_channels, int context_dim, int latent_ch,
                    int latent_hw, int device);
void nope_ldm_destroy(nope_ldm_t* m);
int nope_ldm_load_tensor(nope_ldm_t* m, const char* key, const float* data, const int64_t* shape,
                         int ndim);
int nope_ldm_finalize(nope_ldm_t* m);
int nope_ldm_set_chunk(nope_ldm_t* m, int hyps_per_chunk);       /* ~20.5 MB workspace / hypothesis */
/* conv_impl: 2 = tcgen05 CTA pairs (default), 0 = tcgen05 1-CTA tiles;
 * attn_impl: 0 = tcgen05 attention (default), 1 = CUDA-core twin (bring-up). */
int nope_ldm_set_impl(nope_ldm_t* m, int conv_impl, int attn_impl);
/* Named switches (bring-up / A-B measurements): "fuse_geglu" (default 1: GEGLU runs in the
 * epilogue of its projection GEMM; 0: separate elementwise kernel), "hoist" (default 1: the
 * pose-independent prefix -- input conv, first ResBlock, first transformer up to its
 * self-attention -- runs once per reference instead of once per hypothesis); before
 * nope_ldm_finalize only: "wide_tiles" (default 1: 256-channel GEMM tiles on the CTA-pair kernel),
 * "fold_residual" (default 1: residual adds ride in the GEMM as identity K-segments fed by TMA;
 * 0: added in the epilogue from global memory), "precision" (default 0: fp16 weights; 1: exact
 * weights -- packed rows hold [W_hi | W_lo] and every GEMM accumulates A W_hi + A W_lo, 2x the MMA
 * work; embeddings 1.1e-3 -> below the 1e-3 bar against the fp32 reference). */
int nope_ldm_set_option(nope_ldm_t* m, const char* name, int value);
int nope_ldm_sweep(nope_ldm_t* m, const float* ref_latent, const float* poses, int B, int N,
                   const float* query_latent, float* out_emb, float* out_sim, int k,
                   float* out_topv, int64_t* out_topi, int64_t idx_base, void* stream);
int64_t nope_ldm_last_launch_count(const nope_ldm_t* m);
/* Profiling hook (bench.py roofline), as nope_unet_profile: CUDA events around every tensor-core
 * GEMM / convolution launch (index 0) and every attention launch (index 1) of later sweeps.
 * nope_ldm_profile_read fills ms[2], flops[2] (algorithmic, 2*M*N*K resp. 4*n^2*C per image),
 * launches[2] and synchronises the device. */
int nope_ldm_profile(nope_ldm_t* m, int enable);
int nope_ldm_profile_read(nope_ldm_t* m, double* ms, double* flops, int64_t* launches);
/* Debug: as nope_unet_debug_tap; tap names follow the reference's module paths
 * ("input_blocks.4.0" = ResBlock output, "input_blocks.4" = block output, "middle_block.1",
 * "output_blocks.2.1", "output_blocks.2", ...). */
int nope_ldm_debug_tap(nope_ldm_t* m, const float* ref_latent, const float* poses, int N,
                       const char* tap, float* out, int64_t out_capacity_floats, int* out_C,
                       int* out_H, void* stream);
/* Debug / parity: run ONE module in isolation on fp32 NCHW device inputs.
 *   name "<prefix>.0" of a ResBlock, "<prefix>.1" of a SpatialTransformer (poses [n, 6] needed),
 *   "input_blocks.<i>.0.op" (Downsample), "output_blocks.<i>.2.conv" (Upsample; S = input side).
 *   x0 [n, C0, S, S], x1 (optional, concatenated after x0) [n, C1, S, S] -> out fp32 NCHW.
 * Synchronises the stream. */
int nope_ldm_run_block(nope_ldm_t* m, const char* name, const float* x0, int C0, const float* x1,
                       int C1, int S, int n, const float* poses, float* out, void* stream);
/* Multi-head self-attention core (ldm/attention.py:177-194, heads of 32 channels):
 * qkv [n_img, n_tok, 3C] fp32 (q | k | v) -> out [n_img, n_tok, C] fp32.  impl as attn_impl. */
int nope_op_mh_attention(int impl, const float* qkv, float* out, int n_img, int n_tok, int C,
                         void* stream);

/* ---- VSD evaluation (src/poses/vsd.py, vsd_utils.py; the tless_<cat> branch of model.py:391-541) ----
 * Mesh table: vertices [sum V, 3] fp32 and faces [sum F, 3] int32 (indices local to their mesh) of M
 * meshes packed back to back; mesh_voff / mesh_foff (HOST, int64 [M + 1], starting at 0) delimit them.
 * Render p draws mesh mesh_ids[p] (HOST, int32 [P]) under poses [P, 3, 4] fp32 (R | t, object -> OpenCV
 * camera: x right, y down, z forward) with intrinsics [P, 4] float64 (fx, fy, cx, cy).  Pixel (x, y)
 * samples the image point (x + 0.5, y + 0.5); depth [P, H, W] fp32 is the camera z of the nearest
 * surface with znear <= z <= zfar, 0 where nothing is hit.  No back-face culling.  Renders are
 * bit-reproducible and independent of how they are grouped into calls.
 * nope_vsd_workspace_bytes returns the device workspace nope_vsd_render needs (negative on error). */
int64_t nope_vsd_workspace_bytes(const int64_t* mesh_voff, const int64_t* mesh_foff, int M, const int* mesh_ids,
                                 int P);
int nope_vsd_render(const float* verts, const int* faces, const int64_t* mesh_voff, const int64_t* mesh_foff, int M,
                    const int* mesh_ids, const float* poses, const double* intrinsics, int P, int H, int W,
                    float znear, float zfar, void* workspace, int64_t workspace_bytes, float* depth, void* stream);
/* VSD errors of F frames x k hypotheses (vsd_obj, vsd.py:58-136, bop19 visibility, step cost):
 *   depth_raw [F, H, W] uint16 sensor depth, divided by depth_scale in float64 (T-LESS: 10.0 -> mm);
 *   intrinsics [F, 4] float64 (fx, fy, cx, cy); depth_gt [F, H, W] and depth_est [F, k, H, W] fp32 renders.
 * out_counts [F, k, 3] int64 = (|union|, |intersection|, pixels of the intersection with cost 1);
 * out_err [F, k] float64 = (costs + |union| - |inter|) / |union|, 1.0 when the union is empty. */
int nope_vsd_error(const uint16_t* depth_raw, double depth_scale, const double* intrinsics, const float* depth_gt,
                   const float* depth_est, int F, int k, int H, int W, float delta, double tau, int64_t* out_counts,
                   double* out_err, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NOPE_B200_H */
