/*
 * cdx.h -- C ABI of libcdx.so, the B200-native CycleDiffusion sampling engine.
 *
 * This is the drop-in boundary for the one hot path of ChenWu98/cycle-diffusion: the DPM-Encoder
 * inversion + decode-with-recovered-noise loops including the U-Net / VAE forwards.  Every entry
 * point cites the reference interface it replaces (paths relative to the reference repo root;
 * SDW = model/gan_wrapper/stable_diffusion_stochastic_text_wrapper.py,
 * DW  = model/gan_wrapper/ddpm_ddim_wrapper.py,
 * DDIM = model/lib/stable_diffusion/ldm/models/diffusion/ddim.py,
 * OAI = model/lib/stable_diffusion/ldm/modules/diffusionmodules/openaimodel.py,
 * AEM = model/lib/stable_diffusion/ldm/modules/diffusionmodules/model.py,
 * IU  = model/lib/ddpm_ddim/models/improved_ddpm/unet.py).
 *
 * Conventions
 *   - plain pointers and sizes only; no torch types.  All tensors are fp32.
 *   - "dev" pointers are CUDA device pointers owned by the caller (e.g. torch.Tensor.data_ptr()),
 *     never retained past the call.  Image / latent tensors at the boundary are NCHW contiguous,
 *     exactly the reference's layout; the engine converts to its internal NHWC layout itself.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).  No call synchronises
 *     the device; every call only enqueues work on `stream` (weight loading excepted).
 *   - every function returns 0 on success, a negative CDX_E_* code otherwise; cdx_last_error()
 *     returns a human-readable message for the calling thread's last failure.
 *   - an engine is bound to one device and is NOT thread-safe; use one engine per device/rank.
 */
#ifndef CDX_H_
#define CDX_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CDX_ABI_VERSION 2

#define CDX_OK 0
#define CDX_E_INVALID (-1)   /* bad argument / precondition (the reference's assert) */
#define CDX_E_CUDA (-2)      /* CUDA runtime error */
#define CDX_E_STATE (-3)     /* call order (e.g. forward before finalize) */
#define CDX_E_NOMEM (-4)

typedef struct cdx_engine cdx_engine;
typedef struct cdx_net cdx_net;

/* ---------------------------------------------------------------- engine ------------------- */
int cdx_abi_version(void);
const char* cdx_last_error(void);
/* Creates the per-device context (workspace arena, SM count).  Fails with CDX_E_CUDA when no CUDA
 * device is usable: there is no CPU fallback. */
int cdx_engine_create(int device, cdx_engine** out);
void cdx_engine_destroy(cdx_engine* e);
/* bytes currently reserved by the activation arena (for reporting) */
size_t cdx_engine_workspace_bytes(const cdx_engine* e);
/* number of kernels this engine has launched since creation (bench.py's gpu_launches) */
uint64_t cdx_engine_launch_count(const cdx_engine* e);
/* Per-kernel-family timing with CUDA events on the launching stream (off by default; bench.py turns it on for a
 * separate, untimed pass).  Tags: 0 conv3x3 FFMA, 1 dense FFMA, 2 batched (attention) FFMA, 3 conv3x3 tcgen05,
 * 4 dense tcgen05, 5 batched tcgen05, 6 GroupNorm, 7 LayerNorm, 8 softmax, 9 other.  profile_read synchronises the
 * device, sums the records of `tag` (ms, algorithmic flops / bytes, launches) and keeps them until profile(e, 1/0)
 * is called again. */
#define CDX_PROF_NTAGS 10
int cdx_engine_profile(cdx_engine* e, int enable);
int cdx_engine_profile_read(cdx_engine* e, int tag, double* ms, double* flops, double* bytes, uint64_t* launches);
/* select the dense-contraction path:
 *   0 = SIMT fp32 FFMA tiles (exact fp32)
 *   1 = tcgen05, fp32-faithful split products (default): weight GEMMs / convs as 3 x kind::f16 over an fp16 hi/lo split of
 *       power-of-two-scaled operands, attention and activation x activation contractions as 3 x kind::tf32
 *   2 = as 1 but attention unfused (A/B comparisons)
 *   3 = as 1 with every contraction as 3 x kind::tf32 (the round-1 scheme)
 *   4 = FAST PATH, not fp32-faithful: weight GEMMs / convs with the hi*hi term only (plain fp16 inputs, fp32 accumulate);
 *       reported separately by bench.py together with its measured |delta pixel| */
int cdx_engine_set_mma_mode(cdx_engine* e, int mode);

/* ---------------------------------------------------------------- networks ----------------- */
#define CDX_UNET_OPENAI 1 /* SD v1 / LDM text2img U-Net: OAI:413-742 + attention.py:152-261 */
#define CDX_UNET_IDDPM 2  /* improved-DDPM pixel U-Net: IU:401-668 */
#define CDX_UNET_DDPM 3   /* Ho et al. DDPM pixel U-Net (CelebA-HQ / LSUN checkpoints, DW:360-369): models/ddpm/diffusion.py:192-337 --
                             ResnetBlock + single-head AttnBlock (GroupNorm eps 1e-6, swish), [sin | cos] timestep embedding, conv
                             down / up sampling (asymmetric pad), num_res_blocks + 1 decoder blocks per level (SURVEY 8f-4) */

typedef struct cdx_unet_config {
  int kind;                /* CDX_UNET_* */
  int in_channels, out_channels, model_channels, num_res_blocks;
  int n_mult;
  int channel_mult[8];
  int n_attn;
  int attention_ds[8];     /* downsample factors at which attention runs (OAI:541 / IU:506) */
  int num_heads;           /* OPENAI: heads (d_head = ch / heads, legacy=False, OAI:542-549) */
  int num_head_channels;   /* IDDPM: channels per head (IU:287-293) */
  int context_dim;         /* OPENAI: cross-attention context width (768 SD, 1280 LDM); 0 = the unconditional LDM U-Net
                              (use_spatial_transformer=False, OAI:560-577): attention layers are AttentionBlock + QKVAttentionLegacy
                              (OAI:278-351) with num_head_channels (or num_heads) and the forward takes no context */
} cdx_unet_config;

typedef struct cdx_vae_config { /* AutoencoderKL ddconfig, v1-inference.yaml:51-65 */
  int ch;
  int n_mult;
  int ch_mult[8];
  int num_res_blocks;
  int in_channels, out_ch, z_channels, embed_dim;
  /* vq != 0: VQModelInterface first stage of the unconditional LDMs (ldm/models/autoencoder.py:14-21, 258-282; SURVEY 8f-4): encoder
     -> quant_conv gives h [B, embed_dim, h, w] (no moments, no quantisation on the way in); decode = nearest code of the n_embed x
     embed_dim codebook `quantize.embedding.weight` (taming VectorQuantizer2.forward: argmin of |z|^2 + |e|^2 - 2 z.e, straight-through
     value z + (z_q - z)) -> post_quant_conv -> decoder */
  int vq, n_embed;
} cdx_vae_config;

typedef struct cdx_text_config { /* CLIP ViT-L/14 text tower as FrozenCLIPEmbedder uses it (SURVEY 8f-1): HF CLIPTextModel
                                    "openai/clip-vit-large-patch14": 12 layers, width 768, 12 heads, 77 positions, quick-GELU */
  int vocab_size, width, layers, heads, max_len, mlp_width;
  int kind;     /* CDX_TEXT_CLIP (0 also accepted) or CDX_TEXT_XTRANSFORMER: the LDM BERTEmbedder's in-tree encoder
                   (encoders/modules.py:79-98 -> x_transformer.py TransformerWrapper(Encoder(dim, depth))): pre-LN blocks of
                   bias-free q/k/v (heads x dim_head), full attention, exact-GELU feed-forward; 30522 BERT word pieces */
  int dim_head; /* XTRANSFORMER: per-head width (x_transformer DEFAULT_DIM_HEAD = 64; heads * dim_head may differ from width) */
  /* DirectionalCLIP towers (SURVEY 8f-3; model/energy/clean_clip.py:7-41 runs OpenAI CLIP ViT-B/32 encode_image / encode_text):
     proj_dim > 0 adds the projection head (text: `text_projection.weight` [proj, width], applied to the EOT token's final-LN
     state; vision: `visual_projection.weight`).  kind CDX_CLIP_VISION: the ViT image tower, `patch` x `patch` patches of an
     `image_size`^2 input (HF CLIPVisionModel names under `vision_model.`; vocab_size / max_len unused) */
  int proj_dim, patch, image_size;
} cdx_text_config;
#define CDX_TEXT_CLIP 1
#define CDX_TEXT_XTRANSFORMER 2
#define CDX_CLIP_VISION 3

/* Build the host-side execution plan and parameter inventory (no GPU work). */
int cdx_unet_create(cdx_engine* e, const cdx_unet_config* cfg, cdx_net** out);
int cdx_vae_create(cdx_engine* e, const cdx_vae_config* cfg, cdx_net** out);
/* Text tower; parameter names are HF CLIPTextModel's (text_model.embeddings.token_embedding.weight, ...), i.e. the SD
 * checkpoint's cond_stage_model.transformer.* keys with that prefix stripped. */
int cdx_text_create(cdx_engine* e, const cdx_text_config* cfg, cdx_net** out);
void cdx_net_destroy(cdx_net* n);

/* Parameter inventory in the reference checkpoint's own key names (SURVEY.md Appendix C), so a
 * loader can walk torch.load(ckpt)["state_dict"] (txt2img.py:27-32; DW:378-379). */
int cdx_net_num_params(const cdx_net* n);
const char* cdx_net_param_name(const cdx_net* n, int i);
int cdx_net_param_shape(const cdx_net* n, int i, int64_t dims[4]); /* returns rank */
/* Copy one parameter (host or device fp32, dense, reference layout e.g. OIHW) into the engine. */
int cdx_net_load_param(cdx_net* n, const char* name, const float* data, int data_on_device,
                       const int64_t* dims, int rank);
/* All parameters present -> repack (conv3x3 OIHW -> O,kh,kw,I; split hi/lo planes for 3xTF32). */
int cdx_net_finalize(cdx_net* n);
/* The packed device blob holding every weight of this net; valid after the first load_param.
 * Multi-GPU: rank 0 loads + finalizes, every rank calls cdx_net_adopt_blob() after receiving the
 * blob with one ncclBroadcast (the only collective on the path; replaces the per-process
 * torch.load of txt2img.py:25-42 / DW:378-379). */
int cdx_net_weight_blob(cdx_net* n, void** dev_ptr, size_t* bytes);
int cdx_net_adopt_blob(cdx_net* n); /* mark a blob filled externally (broadcast) as finalized */
/* Sinusoid frequency table for timestep_embedding (util.py:152-172 / nn.py:103-121): the host
 * passes the table computed with the reference expression so that CPU oracle and engine agree
 * bit-for-bit on the frequencies; `half` must equal model_channels/2. */
int cdx_unet_set_time_freqs(cdx_net* n, const float* freqs_host, int half);

/* UNetModel.forward (OAI:710-742 via LatentDiffusion.apply_model ddpm.py:882-983 / IU:639-668).
 * x, out: [B, C, H, W] NCHW dev; t_dev: [B] float timesteps on device (the reference's int64
 * timesteps are cast with .float() at util.py:165); ctx_dev: [B, ctx_len, context_dim] or NULL
 * (IDDPM).  out has out_channels channels (IDDPM: 6 = eps | sigma). */
int cdx_unet_forward(cdx_net* n, const float* x_dev, const float* t_dev, const float* ctx_dev,
                     int ctx_len, float* out_dev, int B, int H, int W, void* stream);

/* AutoencoderKL.encode (autoencoder.py:324-328 + AEM:434-459): img [B,3,R,R] in [-1,1] ->
 * moments [B, 2*embed_dim, R/8, R/8] (mean | logvar), both NCHW dev. */
int cdx_vae_encode(cdx_net* n, const float* img_dev, float* moments_dev, int B, int R, void* stream);
/* FrozenCLIPEmbedder.forward after tokenisation (ldm/modules/encoders/modules.py:140-158 -> transformer(input_ids=tokens)
 * .last_hidden_state; HF modeling_clip.py CLIPTextTransformer.forward, transformers==4.19.2 pinned by environment.yml:466):
 * token + position embedding, `layers` pre-LN blocks with causal self-attention and quick-GELU MLP, final LayerNorm.
 * ids_dev [B, L] int32 token ids (L <= max_len); out_dev [B, L, width] fp32.
 * kind XTRANSFORMER: BERTEmbedder.forward after tokenisation = transformer(tokens, return_embeddings=True)
 * (x_transformer.py:598-626, 481-523): parameter names transformer.token_emb.weight, transformer.attn_layers.layers.N.* ... */
int cdx_text_encode(cdx_net* n, const int* ids_dev, int B, int L, float* out_dev, void* stream);
/* AutoencoderKL.decode (autoencoder.py:330-333 + AEM:535-568): z [B,embed_dim,h,h] (already
 * divided by scale_factor) -> img [B, out_ch, 8h, 8h]. */
int cdx_vae_decode(cdx_net* n, const float* z_dev, float* img_dev, int B, int h, void* stream);

/* ---------------------------------------------------------------- per-step kernels ---------- */
/* All element counts `n` are B*C*H*W of one NCHW tensor; scalars are the batch-uniform fp32
 * coefficients the reference broadcasts as [B,1,1,1] tensors.  Arithmetic is done op-by-op with
 * round-to-nearest (no FMA contraction) in the reference's evaluation order, so these are
 * bit-exact against the reference CPU path on identical inputs. */

/* out = a*x + b  (image normalisation SDW:176 / DW:470, post-process SDW:135-137, 1/scale_factor) */
int cdx_affine(cdx_engine* e, const float* x, float a, float b, float* out, size_t n, void* stream);
/* out = (x + b) * a   ((image - 0.5) * 2.0, exact reference order) */
int cdx_shift_scale(cdx_engine* e, const float* x, float b, float a, float* out, size_t n, void* stream);
/* x_t = sqrt_a*x0 + sqrt_1ma*noise  (DDIM:477-479 / DW:310-314) */
int cdx_q_sample(cdx_engine* e, const float* x0, const float* noise, float sqrt_a, float sqrt_1ma,
                 float* out, size_t n, void* stream);
/* DiagonalGaussianDistribution.sample * scale_factor (distributions.py:24-37, ddpm.py:536-543):
 * moments [B,2C,h,w]; noise [B,C,h,w] or NULL for the posterior mean (latentdiff copy). */
int cdx_vae_posterior(cdx_engine* e, const float* moments, const float* noise, float scale_factor,
                      float* out, int B, int C, int hw, void* stream);

typedef struct cdx_ddim_coef { /* one DDIM step, fp32 scalars exactly as ddim.py:570-573 builds them */
  float sqrt_at;        /* a_t.sqrt() */
  float sqrt_1m_at;     /* (1 - a_t).sqrt()                 -- sample_xt_next, ddim.py:597 */
  float sqrt_1m_at_tab; /* ddim_sqrt_one_minus_alphas[index] -- compute_eps, ddim.py:573 */
  float sqrt_aprev;     /* a_prev.sqrt() */
  float dir_coef;       /* (1 - a_prev - sigma_t**2).sqrt() */
  float sigma;          /* sigma_t */
} cdx_ddim_coef;

/* DDIMSampler.sample_xt_next (ddim.py:582-601): posterior sample x_{t-1} | x_t, x0 */
int cdx_ddim_posterior_sample(cdx_engine* e, const float* x0, const float* xt, const float* noise,
                              const cdx_ddim_coef* c, float* xt_next, size_t n, void* stream);
/* CFG combine + DDIMSampler.compute_eps tail (ddim.py:555-559, 575-579).  e_uc may be NULL
 * (scale 1 -> e_c only, ddim.py:550-551). */
int cdx_ddim_compute_eps(cdx_engine* e, const float* xt, const float* xt_next, const float* e_c,
                         const float* e_uc, float scale, const cdx_ddim_coef* c, float* eps_out,
                         size_t n, void* stream);
/* CFG combine + DDIMSampler.p_sample_ddim_with_eps tail (ddim.py:613-617, 634-645). */
int cdx_ddim_step_with_eps(cdx_engine* e, const float* x, const float* e_c, const float* e_uc,
                           float scale, const float* eps, const cdx_ddim_coef* c, float* x_prev,
                           size_t n, void* stream);

typedef struct cdx_pixel_coef { /* one step of the pixel-space samplers, DW:114-307 */
  int ddpm;           /* 1 = sample_type 'ddpm', 0 = 'ddim' */
  float sqrt_at;      /* at.sqrt() */
  float sqrt_1m_at;   /* (1 - at).sqrt() */
  float sqrt_at_next; /* at_next.sqrt() */
  float c1, c2;       /* ddim: eta*sqrt((1-at/at_next)(1-at_next)/(1-at)), sqrt((1-at_next)-c1^2) */
  float w0, wt, post_std;   /* ddpm posterior q(x_{t-1}|x_t,x0): DW:291-298 */
  float weight, inv_sqrt_1m_bt, std_model, mask; /* ddpm model mean / exp(0.5 logvar): DW:202-210 */
} cdx_pixel_coef;

/* sample_xt_next (DW:283-307) */
int cdx_pixel_posterior_sample(cdx_engine* e, const float* x0, const float* xt, const float* noise,
                               const cdx_pixel_coef* c, float* xt_next, size_t n, void* stream);
/* compute_eps (DW:230-280); et: U-Net output [B,Cnet,H,W] of which the first C channels are used
 * (learn_sigma split, DW:236-238); chw = C*H*W, net_chw = Cnet*H*W */
int cdx_pixel_compute_eps(cdx_engine* e, const float* xt, const float* xt_next, const float* et,
                          const cdx_pixel_coef* c, float* eps_out, int B, int chw, int net_chw,
                          void* stream);
/* denoising_step_with_eps / denoising_step (DW:114-227, diffusion_utils.py:23-136) */
int cdx_pixel_step_with_eps(cdx_engine* e, const float* xt, const float* et, const float* eps,
                            const cdx_pixel_coef* c, float* xt_next, int B, int chw, int net_chw,
                            void* stream);

/* ---------------------------------------------------------------- loop drivers -------------- */
/* DDIMSampler._ddpm_ddim_encoding (ddim.py:450-501), all refine steps on `stream`, no host sync.
 *   x0      [B,C,h,w]        clean latent
 *   c, uc   [B,L,D]          conditioning / unconditional conditioning (uc may be NULL if scale==1)
 *   coef    host[n_steps]    loop order (i = 0 is the noisiest step, index = n_steps-1)
 *   t_host  host[n_steps]    timestep value fed to the U-Net at iteration i
 *   n_rec                    number of steps that recover noise (min(n_steps, white_box-skip-1))
 *   noise   [n_rec(+1 incl. x_T draw), B,C,h,w] dev: noise[0] = x_T draw, noise[1+i] = draw of
 *                            iteration i (unused when index==0, ddim.py:583-584)
 *   sqrt_a_T, sqrt_1ma_T     at.sqrt(), (1-at).sqrt() of ddim.py:478-479
 *   z_out   [B, n_rec+1, C,h,w]  = stack(z_list, dim=1) (SDW:203)
 */
int cdx_latent_encode(cdx_net* unet, const float* x0, const float* c, const float* uc, int ctx_len,
                      float scale, const cdx_ddim_coef* coef, const float* t_host, int n_steps,
                      int n_rec, const float* noise, float sqrt_a_T, float sqrt_1ma_T, float* z_out,
                      int B, int C, int h, int w, void* stream);
/* DDIMSampler.ddim_sampling_with_eps (ddim.py:395-448): z [B, n_eps+1, C,h,w] (x_T first, SDW:150-154);
 * extra_noise [n_steps-n_eps, B,C,h,w] for steps without recovered noise (may be NULL if none). */
int cdx_latent_decode(cdx_net* unet, const float* z, int n_eps, const float* c, const float* uc,
                      int ctx_len, float scale, const cdx_ddim_coef* coef, const float* t_host,
                      int n_steps, const float* extra_noise, float* x_out, int B, int C, int h, int w,
                      void* stream);
/* Both chains in lock-step (SURVEY.md 7 step 8 / 8b; the loop shape of Diffusers' CycleDiffusionPipeline.__call__): the source chain
 * of _ddpm_ddim_encoding (ddim.py:450-501) under c_src / src_scale and the target chain of ddim_sampling_with_eps (ddim.py:395-448)
 * under c_tgt / tgt_scale advance together, ONE U-Net call per step on the batch [source segments | target segments] (B rows per
 * segment; a chain contributes [uncond, cond] when its scale is neither 0 nor 1), and the noise recovered at step i is consumed by the
 * target chain inside the same fused elementwise kernel: no z buffer.  Requires all n_steps noises to be recoverable
 * (white_box_steps > custom_steps - skip); noise [n_steps+1, B,C,h,w] as for cdx_latent_encode.  z_out (optional, may be NULL)
 * receives [B, n_steps+1, C,h,w] exactly as cdx_latent_encode would produce it.  Per-sample results equal the two-phase
 * cdx_latent_encode + cdx_latent_decode up to the summation order of split-K GEMMs (the batch size differs). */
int cdx_cycle_lockstep(cdx_net* unet, const float* x0, const float* c_src, const float* c_tgt, const float* uc,
                       int ctx_len, float src_scale, float tgt_scale, const cdx_ddim_coef* coef,
                       const float* t_host, int n_steps, const float* noise, float sqrt_a_T,
                       float sqrt_1ma_T, float* x_out, float* z_out, int B, int C, int h, int w,
                       void* stream);
/* cdx_cycle_lockstep for a source and a target network (two unconditional LDMs, latentdiff_stochastic_wrapper.py:253-311: the
 * DPM-Encoder of one model, ddim.py:450-501, feeding the decode of the other, ddim.py:395-448, as one loop).  Same arguments and
 * loop as cdx_cycle_lockstep, but each step makes two U-Net calls: the source segments through src_unet and the target segments
 * through tgt_unet, each chain at the batch it has in cdx_latent_encode / cdx_latent_decode, so the result (and z_out) equals the
 * two-phase cdx_latent_encode(src_unet) + cdx_latent_decode(tgt_unet) bit for bit.  Context-free U-Nets pass c_src = c_tgt = uc =
 * NULL and ctx_len = 0.  The two networks may belong to different engines on the same device: both workspaces are sized and both
 * engines' stream hand-overs are honoured; all work runs on `stream`. */
int cdx_cycle_lockstep_pair(cdx_net* src_unet, cdx_net* tgt_unet, const float* x0, const float* c_src, const float* c_tgt,
                            const float* uc, int ctx_len, float src_scale, float tgt_scale, const cdx_ddim_coef* coef,
                            const float* t_host, int n_steps, const float* noise, float sqrt_a_T,
                            float sqrt_1ma_T, float* x_out, float* z_out, int B, int C, int h, int w,
                            void* stream);
/* The same three loops with PER-SAMPLE guidance scales (device arrays of B floats): the ensemble driver of the text wrappers
 * (SDW:146-165 generate, :189-204 encode -- the reference loops trial x encoder-scale x skip, then x decoder-scale, one chain at a
 * time, recomputing the conditioning and every context K/V projection per member).  Members that share a schedule are batched
 * along B: mode 1 = encode (x0, c_src, src_scales, noise -> z_out), 2 = decode (z_in, c_tgt, tgt_scales -> x_out), 3 = lock-step.
 * Both CFG segments run for every member; a member whose scale is 1 (0) takes eps-hat(c) (eps-hat(uc)) unchanged, exactly the
 * reference's single-forward branch (ddim.py:550-551), so each member equals its own cdx_latent_encode / _decode call.  The context
 * K / V projections are computed once per loop for the whole batch. */
int cdx_latent_loop_ens(cdx_net* unet, int mode, const float* x0, const float* c_src, const float* c_tgt, const float* uc,
                        int ctx_len, const float* src_scales, const float* tgt_scales, const cdx_ddim_coef* coef,
                        const float* t_host, int n_steps, int n_rec, const float* noise, float sqrt_a_T,
                        float sqrt_1ma_T, const float* z_in, int n_eps, const float* extra_noise, float* z_out,
                        float* x_out, int B, int C, int h, int w, void* stream);
/* ---- Directional-CLIP ranking and the evaluation metrics on the device (SURVEY 8f-3)
 * clip_preprocess: clean_clip.py:14-17 = Resize(size, bicubic) + CenterCrop(size) + Normalize(mean, std) on a float image batch in
 *   [0,1] (square inputs; torch bicubic, A = -0.75, align_corners = False, no antialias -- the tensor path of the torchvision release
 *   the reference pins).  img [B,3,R,R] -> out [B,3,size,size].
 * cdx_clip_image_features: CLIP.encode_image = ViT tower -> ln_post(class token) @ proj  -> [B, proj_dim] (net kind CDX_CLIP_VISION).
 * cdx_text_features: CLIP.encode_text = final-LN state at the EOT token (argmax of the ids) @ text_projection -> [B, proj_dim].
 * cdx_dclip_scores: clean_clip.py:24-39: L2-normalise the four feature sets, clip = <img, dec_text>, dclip = <unit(img - orig),
 *   unit(dec_text - enc_text)>.  All [B, D] device arrays; clip_out / dclip_out [B].
 * cdx_image_metrics: evaluation/translate_text.py:76-89 per image pair after clamp(0,1): PSNR = 10 log10(1 / mse) (100 when equal;
 *   evaluation/utils.py:60-66), L2 = sqrt(sum sq diff), SSIM of the x255 images (11x11 Gaussian sigma 1.5, valid region, per channel,
 *   mean of 3; evaluation/utils.py:35-57).  a, b [B,3,H,W] -> out [B,3] = {psnr, ssim, l2} (fp32). */
int cdx_clip_preprocess(cdx_engine* e, const float* img, int B, int R, int size, float* out, void* stream);
int cdx_clip_image_features(cdx_net* vision, const float* pixels, int B, float* out, void* stream);
int cdx_text_features(cdx_net* text, const int* ids_dev, int B, int L, float* out, void* stream);
int cdx_dclip_scores(cdx_engine* e, const float* img_f, const float* orig_f, const float* enc_f, const float* dec_f, int B, int D,
                     float* clip_out, float* dclip_out, void* stream);
int cdx_image_metrics(cdx_engine* e, const float* a, const float* b, int B, int H, int W, float* out, void* stream);
/* DDPMDDIMWrapper.encode loop (DW:483-521): coef/t_host have n_rec entries (loop order);
 * noise[0] = x_T draw, noise[1+i] = draw of iteration i; z_out [B, n_rec+1, C,R,R]. */
int cdx_pixel_encode(cdx_net* unet, const float* x0, const cdx_pixel_coef* coef, const float* t_host,
                     int n_rec, const float* noise, float sqrt_a_T, float sqrt_1ma_T, float* z_out,
                     int B, int C, int R, void* stream);
/* DDPMDDIMWrapper.generate main loop (DW:415-429): n_steps = n_eps + 1 (the last step's noise is
 * multiplied by 0 in the reference; pass it in last_noise or NULL). */
int cdx_pixel_decode(cdx_net* unet, const float* z, int n_eps, const cdx_pixel_coef* coef,
                     const float* t_host, int n_steps, const float* last_noise, float* x_out, int B,
                     int C, int R, void* stream);

/* Two-model pixel cycle as one lock-step loop: DDPMDDIMWrapper.encode of src_unet (DW:483-521) feeding DDPMDDIMWrapper.generate's
 * main loop on tgt_unet (DW:415-429) without a z buffer.  Order of work: x_T = q_sample(x0, noise[0]) with sqrt_a_T / sqrt_1ma_T
 * taken at index n_steps-1 (the DW:483 quirk); the target chain starts from the same x_T; n_steps-1 iterations, each one src_unet
 * forward, one tgt_unet forward and ONE fused kernel (sample_xt_next DW:283-307, compute_eps DW:230-280 on the first C channels
 * of the source output, denoising_step_with_eps DW:114-227 of the target with that noise); then a target-only step for the last
 * (0, -1) pair with last_noise (multiplied by 0, DU:115,131; may be NULL).
 *   coef / t_host  host[n_steps] loop order (noisiest first), shared by both chains
 *   noise          [n_steps, B,C,R,R] dev: noise[0] = x_T draw, noise[1+i] = draw of iteration i (as cdx_pixel_encode)
 *   x_out          [B,C,R,R] target chain result (before shift / scale)
 *   z_out          optional [B, n_steps, C,R,R]: the recovered noise, bit-equal to cdx_pixel_encode's z
 * Each chain runs at batch B on its own network, so x_out equals cdx_pixel_encode(src_unet) + cdx_pixel_decode(tgt_unet) bit for
 * bit.  The networks may belong to different engines on the same device (both workspaces sized, both stream hand-overs honoured);
 * all work runs on `stream`. */
int cdx_pixel_cycle_lockstep(cdx_net* src_unet, cdx_net* tgt_unet, const float* x0, const cdx_pixel_coef* coef,
                             const float* t_host, int n_steps, const float* noise, float sqrt_a_T, float sqrt_1ma_T,
                             const float* last_noise, float* x_out, float* z_out, int B, int C, int R, void* stream);

/* ---------------------------------------------------------------- unit-test hooks ----------- */
/* Individual ops exported for per-op parity tests (tests/test_ops_gpu.py, tests/test_gemm_epilogue_gpu.py).
 * NHWC = [B,H,W,C].  Not part of the drop-in interface: these may change without an ABI version bump. */

/* Which GEMM variant ran (filled on the real pass of the call, host side only). */
#define CDX_GEMM_FFMA 0      /* SIMT fp32 tiles */
#define CDX_GEMM_SS 1        /* tcgen05 3 x kind::tf32, both operands split in the kernel */
#define CDX_GEMM_TS 2        /* tcgen05 3 x kind::tf32 on pre-split weight planes */
#define CDX_GEMM_H16 3       /* tcgen05 3 x kind::f16 fp16-split, single CTA */
#define CDX_GEMM_H16_PAIR 4  /* the same on CTA pairs (cta_group::2) */
typedef struct cdx_gemm_plan {
  int path;          /* CDX_GEMM_* */
  int halo;          /* conv3x3 halo schedule */
  int epi_tma;       /* TMA-store epilogue (else the per-row epilogue, or split-K partials + reduce kernel) */
  int tn_w;          /* tile width along N */
  int splits;        /* split-K factor (> 1: partial sums reduced by a second kernel) */
  int tail16;        /* the TMA epilogue stores some 16-column tail boxes */
  int side_done;     /* bit 0: c_amax produced by the GEMM kernels, bit 1: c_stats produced by the epilogue (else by an extra pass) */
} cdx_gemm_plan;

/* One GEMM with the epilogue options the networks use:
 *   C = alpha * A . W^T (+ bias[n]) (+ rowvec[m / rows_per_batch, n]) (+ residual[m, n])
 * conv = 0: A [M, C1] (optionally | A2 [M, C2], a channel concat), W [N, C1 + C2].
 * conv = 1: A is the implicit im2col of a 3x3 convolution over NHWC x [B, H, W, C1] (stride 1 / 2, `pad` zero rows / columns
 *   before the image -- stride 2 with pad 0 is the VAE's (0,1,0,1) padding -- and nearest `up` x upsampling of the input);
 *   W is OIHW [N, C1, 3, 3]; M = B * Ho * Wo.
 * a_amax / a2_amax: optional device scalars >= max |A| / |A2| (as tracked by a producer); measured by the GEMM when null.
 * geglu: W (and bias) in the reference layout [N/2 value rows; N/2 gate rows]; C [M, N/2] = value * gelu(gate).
 * out_nchw: C stored as [M / rows_per_img, N, rows_per_img].  C_lo: C and C_lo receive the TF32 hi / lo planes of the result.
 * Ct_hi / Ct_lo: columns n >= t_col0 stored transposed as TF32 planes at [(n - t_col0) * ldt + m].
 * c_amax (float) / c_stats (double [M / rows_per_batch, N, 2]): optional device outputs, zeroed here, receive max |stored C| and the
 * per-(image, channel) {sum, sum of squares} of C.  Zero ld* / rows_per_* fields take the dense defaults.
 * plan: optional host output. */
typedef struct cdx_gemm_test {
  int conv;
  int M;                                  /* dense */
  int B, H, W, stride, pad, up;           /* conv */
  int N, C1, C2;
  const float* A; const float* A2;
  const float* a_amax; const float* a2_amax;
  const float* w; const float* bias;
  const float* rowvec; int ld_rowvec; int rows_per_batch;
  const float* residual; int ldr;
  float alpha;
  int geglu;
  float* C; int ldc;
  int out_nchw, rows_per_img;
  float* C_lo;
  float* Ct_hi; float* Ct_lo; int t_col0; long long ldt;
  float* c_amax; double* c_stats;
  cdx_gemm_plan* plan;
} cdx_gemm_test;
int cdx_op_gemm(cdx_engine* e, const cdx_gemm_test* t, void* stream);
/* GroupNorm(32) of x [B,HW,C1] (optionally channel-concatenated with x2 [B,HW,C2]), y = [silu](gn(x) * (1 + scale) + shift) with
 * scale / shift [B, *] rows of stride ld_ss (may be null).  st1 / st2: optional per-(image, channel) {sum, sum of squares} of x / x2
 * (fp64, as a GEMM epilogue produces them), computed here when null.  amax: optional device scalar, receives max |y| (zeroed here). */
int cdx_op_groupnorm(cdx_engine* e, const float* x_nhwc, int C1, const float* x2_nhwc, int C2, const float* gamma,
                     const float* beta, float eps, int silu, const float* scale, const float* shift, int ld_ss,
                     const double* st1, const double* st2, float* amax, float* y_nhwc, int B, int HW, void* stream);
int cdx_op_layernorm(cdx_engine* e, const float* x, const float* gamma, const float* beta, float* y,
                     int M, int C, void* stream);
/* softmax(q k^T * scale) v with q [B,Nq,heads*d], k/v [B,Nk,heads*d] -> [B,Nq,heads*d] */
int cdx_op_attention(cdx_engine* e, const float* q, const float* k, const float* v, float* out, int B,
                     int Nq, int Nk, int heads, int d, float scale, void* stream);
int cdx_op_nchw_to_nhwc(cdx_engine* e, const float* x, float* y, int B, int C, int HW, void* stream);
int cdx_op_nhwc_to_nchw(cdx_engine* e, const float* x, float* y, int B, int C, int HW, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CDX_H_ */
