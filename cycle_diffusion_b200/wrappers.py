"""Drop-in `gan_wrapper` classes: the reference's plugin surface for the hot path, backed by libcdx.

Mirrors (same constructor kwargs, method names, argument meaning, return layouts and precondition checks):
  SDStochasticTextWrapper            ref model/gan_wrapper/stable_diffusion_stochastic_text_wrapper.py:100-253
  LatentDiffStochasticTextWrapper    ref model/gan_wrapper/latentdiff_stochastic_text_wrapper.py:102-252
  DDPMDDIMWrapper                    ref model/gan_wrapper/ddpm_ddim_wrapper.py:317-538
  get_gan_wrapper                    ref model/gan_wrapper/get_gan_wrapper.py:3-31

Differences that are deliberate and documented in INTEGRATION.md:
  * weights come from a reference-format ``state_dict`` / checkpoint path given by keyword (or ``'synthetic'``);
    the packed blob can be shared between wrappers and broadcast across ranks;
  * the text encoder is ``cond_stage(list[str]) -> [B,77,D]``: either an injected callable or the in-engine towers
    (``ClipTextCondStage`` / ``BertTextCondStage``, SURVEY.md 8f-1), which are built automatically from the checkpoint's
    ``cond_stage_model.*`` keys when a host ``tokenizer`` is given.  The deterministic ``SyntheticTextEncoder`` stand-in is
    used ONLY together with ``state_dict='synthetic'``; a real checkpoint without a conditioning model raises;
  * random draws are taken from the torch CPU generator in the reference's order and uploaded, so a run is
    reproducible against the reference CPU path under the same ``torch.manual_seed``;
  * Directional-CLIP ranking of the ensemble is an injected callable (SURVEY.md 8f-3); with a single ensemble
    member no ranking is needed.
"""
import hashlib
import os

import numpy as np
import torch

from . import specs
from .engine import Engine, UNet, VAE
from .schedule import DDIMSchedule, PixelSchedule


class ClipTextCondStage:
    """In-engine conditioning model: drop-in for ``model.get_learned_conditioning`` with FrozenCLIPEmbedder behind it
    (ddpm.py:545-556 -> encoders/modules.py:148-158): ``list[str] -> [B, 77, 768]`` on the engine's device.

    ``tokenizer``: callable ``list[str] -> LongTensor [B, L]`` -- e.g. ``lambda t: hf_tok(t, truncation=True, max_length=77,
    padding='max_length', return_tensors='pt')['input_ids']`` with HF ``CLIPTokenizer`` (the BPE vocabulary is host data and
    not part of the engine).  ``state_dict``: HF CLIPTextModel keys, optionally under ``prefix`` (the SD checkpoint keeps them
    under ``cond_stage_model.transformer.``)."""

    def __init__(self, engine, state_dict, tokenizer, cfg=None, prefix=''):
        from .engine import TextEncoder
        self.cfg = cfg or specs.clip_text_config()
        self.tokenizer = tokenizer
        self.encoder = TextEncoder(engine, self.cfg)
        self.encoder.load_state_dict({k: v for k, v in state_dict.items() if k.startswith(prefix)}, prefix=prefix)

    def __call__(self, texts):
        ids = self.tokenizer(list(texts))
        assert ids.dim() == 2 and ids.shape[0] == len(texts), 'tokenizer must return [B, L] ids'
        return self.encoder(ids)


class BertTextCondStage(ClipTextCondStage):
    """Same for the LDM text2img-large conditioning model: BERTEmbedder (encoders/modules.py:79-102; 32 x 1280 x_transformer
    encoder over BERT word pieces).  ``tokenizer``: e.g. HF ``BertTokenizerFast`` with ``padding='max_length', max_length=77``
    (modules.py:66-72); the LDM checkpoint keeps the weights under ``cond_stage_model.``."""

    def __init__(self, engine, state_dict, tokenizer, cfg=None, prefix=''):
        super().__init__(engine, state_dict, tokenizer, cfg or specs.bert_text_config(), prefix)


class SyntheticTextEncoder:
    """Deterministic stand-in for FrozenCLIPEmbedder / BERTEmbedder: prompt string -> N(0,1) tokens [77, dim].

    Same interface as ``model.get_learned_conditioning`` (ddpm.py:545-556).  Not a language model: it only gives
    distinct, reproducible conditioning tensors so the sampling path can be exercised without checkpoints.
    """

    def __init__(self, dim, n_tokens=77, device='cpu'):
        self.dim, self.n_tokens, self.device = dim, n_tokens, device

    def __call__(self, texts):
        assert isinstance(texts, list) and isinstance(texts[0], str)       # SDW:29-30
        out = []
        for t in texts:
            seed = int.from_bytes(hashlib.sha256(t.encode('utf-8')).digest()[:4], 'little')
            g = torch.Generator().manual_seed(seed)
            out.append(torch.randn(self.n_tokens, self.dim, generator=g))
        return torch.stack(out).to(self.device)


def _load_sd(state_dict, ckpt_default, synth_params, seed):
    if isinstance(state_dict, dict):
        return state_dict
    if state_dict == 'synthetic':
        return specs.synth_state_dict(synth_params, seed)
    path = state_dict if isinstance(state_dict, str) else ckpt_default
    if not os.path.exists(path):
        raise FileNotFoundError(f'checkpoint {path} not found; pass state_dict=<dict>, a path, or "synthetic"')
    sd = torch.load(path, map_location='cpu')
    return sd['state_dict'] if 'state_dict' in sd else sd       # txt2img.py:27-32 / DW:378-379


class _LatentGenerator:
    """What the text wrappers call ``self.generator`` (LatentDiffusion): U-Net + first stage + cond stage."""

    def __init__(self, engine, unet, vae, cond_stage, channels, image_size, scale_factor, sample_posterior):
        self.engine, self.unet, self.vae, self.cond_stage = engine, unet, vae, cond_stage
        self.channels, self.image_size, self.scale_factor = channels, image_size, scale_factor
        self.sample_posterior = sample_posterior
        self.alphas_cumprod = None      # default LDM linear schedule (v1-inference.yaml:5-9)

    def get_learned_conditioning(self, c):
        return self.cond_stage(c)

    def encode_first_stage(self, image):
        return self.vae.encode_moments(image)                              # moments of the DiagonalGaussianDistribution

    def get_first_stage_encoding(self, moments):
        if self.vae.cfg.get('vq'):                                         # VQModelInterface: the encoder output itself (ddpm.py:536-543, tensor branch)
            return self.engine.affine(moments, self.scale_factor, 0.0)
        noise = None
        if self.sample_posterior:                                          # ddpm.py:536-543; distributions.py:36 draws on the CPU
            B, C2, h, w = moments.shape
            noise = torch.randn(B, C2 // 2, h, w)
        return self.engine.vae_posterior(moments, noise, self.scale_factor)

    def decode_first_stage(self, z):
        return self.vae.decode(self.engine.affine(z, 1. / self.scale_factor, 0.0))     # ddpm.py:705


class _StochasticTextWrapperBase(torch.nn.Module):
    RESOLUTION = 512
    LATENT = 64
    CONTEXT_DIM = 768
    SAMPLE_POSTERIOR = True
    CKPT_DIR = 'ckpts/stable_diffusion'
    COND_PREFIX = 'cond_stage_model.transformer.'     # FrozenCLIPEmbedder.transformer (encoders/modules.py:140-146)
    COND_CLASS = ClipTextCondStage

    @classmethod
    def default_checkpoint(cls, source_model_type):
        """SDW:21-23: ``ckpts/stable_diffusion/<source_model_type>``."""
        return os.path.join(cls.CKPT_DIR, str(source_model_type))

    def __init__(self, source_model_type, custom_steps, eta, white_box_steps, skip_steps,
                 encoder_unconditional_guidance_scales=None, decoder_unconditional_guidance_scales=None, n_trials=None, *,
                 engine=None, device=0, state_dict=None, cond_stage=None, ranker=None, unet_config=None, vae_config=None,
                 latent_size=None, resolution=None, generator=None, seed=1234, tokenizer=None, ensemble_batch=16):
        super().__init__()
        # ensemble members that share a schedule are batched along the batch dimension, up to this many samples per sampling loop
        # (cdx_latent_loop_ens); None / 0 = one member at a time, the reference's loop shape
        self.ensemble_batch = ensemble_batch
        self.encoder_unconditional_guidance_scales = encoder_unconditional_guidance_scales
        self.decoder_unconditional_guidance_scales = decoder_unconditional_guidance_scales
        self.n_trials = n_trials
        self.eta, self.custom_steps, self.white_box_steps, self.skip_steps = eta, custom_steps, white_box_steps, skip_steps
        self.resolution = resolution or self.RESOLUTION
        self.precision = "full"
        self.directional_clip = ranker
        if generator is not None:
            self.generator = generator
            self.engine = generator.engine
        else:
            self.engine = engine or Engine(device)
            ucfg = unet_config or specs.sd_unet_config(self.CONTEXT_DIM)
            vcfg = vae_config or specs.kl_f8_config()
            unet, vae = UNet(self.engine, ucfg, 'openai'), VAE(self.engine, vcfg)
            ckpt = self.default_checkpoint(source_model_type)
            cond = cond_stage
            if state_dict == 'synthetic':
                unet.load_state_dict(specs.synth_state_dict(specs.openai_unet_params(ucfg), seed))
                vae.load_state_dict(specs.synth_state_dict(specs.kl_vae_params(vcfg), seed + 1))
                if cond is None:
                    cond = SyntheticTextEncoder(ucfg['context_dim'])        # random-init weights: random (but reproducible) conditioning
            else:
                sd = _load_sd(state_dict, ckpt, None, seed)
                unet.load_state_dict(sd, prefix='model.diffusion_model.', strict=False)
                vae.load_state_dict(sd, prefix='first_stage_model.', strict=False)
                if cond is None:
                    # the reference builds the conditioning model from the same checkpoint (txt2img.py:27-45); do the same, and never
                    # fall back silently to noise tokens when real weights were loaded
                    has_tower = any(k.startswith(self.COND_PREFIX) for k in sd)
                    if tokenizer is not None and has_tower:
                        cond = self.COND_CLASS(self.engine, sd, tokenizer, prefix=self.COND_PREFIX)
                    else:
                        raise ValueError(
                            f'{type(self).__name__}: a checkpoint was loaded but no conditioning model is available '
                            f'({"no " + self.COND_PREFIX + "* keys in the checkpoint" if not has_tower else "no tokenizer= given"}). '
                            'Pass cond_stage=<callable list[str] -> [B,77,D]> or tokenizer=<callable list[str] -> ids [B,L]> '
                            '(the in-engine text tower is then built from the checkpoint).')
            self.generator = _LatentGenerator(self.engine, unet, vae, cond, ucfg['in_channels'], latent_size or self.LATENT, 0.18215,
                                              self.SAMPLE_POSTERIOR)
        self._dummy = torch.nn.Parameter(torch.zeros(1, device=self.engine.device), requires_grad=False)

    # -- helpers mirroring the module-level functions of the reference wrapper
    def _get_condition(self, text, bs):
        assert isinstance(text, list)
        assert isinstance(text[0], str)
        uc = self.generator.get_learned_conditioning(bs * [""])
        c = self.generator.get_learned_conditioning(text)
        return c, uc

    def _encode_noise(self, sched, n_rec, shape):
        """Draws of _ddpm_ddim_encoding in order: x_T (ddim.py:479), then one per step except index==0 (ddim.py:583-584, 599)."""
        noise = torch.zeros((n_rec + 1,) + tuple(shape))
        noise[0] = torch.randn(shape)
        for i in range(n_rec):
            if sched.refine_steps - 1 - i != 0:
                noise[1 + i] = torch.randn(shape)
        return noise

    def _chunks(self, members, bsz):
        per = max(1, (self.ensemble_batch or 1) // max(1, bsz))
        return [members[i:i + per] for i in range(0, len(members), per)]

    def _generate_batched(self, z_ensemble, decode_text):
        """generate() with the members of one schedule batched along B: the conditioning is computed once, the context K / V
        projections once per loop, and (member, scale) pairs share U-Net calls.  Random draws (ddim.py:640) keep the reference order."""
        g = self.generator
        bsz = z_ensemble[0].shape[0]
        c, uc = self._get_condition(decode_text, bsz)
        nsc = len(self.decoder_unconditional_guidance_scales)
        imgs = [None] * (len(z_ensemble) * nsc)
        jobs = {}                                         # skip -> [(output slot, eps_list, scale, extra)]
        for i, z in enumerate(z_ensemble):
            skip_steps = self.skip_steps[i % len(self.skip_steps)]
            if self.white_box_steps != -1:
                eps_list = z.view(bsz, (self.white_box_steps - skip_steps), g.channels, g.image_size, g.image_size)
            else:
                eps_list = z.view(bsz, 1, g.channels, g.image_size, g.image_size)
            sched = DDIMSchedule(self.custom_steps, self.eta, skip_steps, g.alphas_cumprod)
            n_extra = sched.refine_steps - (eps_list.shape[1] - 1)
            for k, scale in enumerate(self.decoder_unconditional_guidance_scales):
                extra = torch.stack([torch.randn(eps_list[:, 0].shape) for _ in range(n_extra)]) if n_extra > 0 else None
                jobs.setdefault(skip_steps, []).append((i * nsc + k, eps_list, float(scale), extra))
        for skip_steps, members in jobs.items():
            sched = DDIMSchedule(self.custom_steps, self.eta, skip_steps, g.alphas_cumprod)
            for chunk in self._chunks(members, bsz):
                zc = torch.cat([m[1].to(self.engine.device) for m in chunk], dim=0)
                sc = torch.tensor([m[2] for m in chunk for _ in range(bsz)])
                ex = torch.cat([m[3] for m in chunk], dim=1) if chunk[0][3] is not None else None
                rep = len(chunk)
                sample = g.unet.latent_decode_ens(zc, c.repeat(rep, 1, 1), uc.repeat(rep, 1, 1), sc, sched, ex)
                dec = g.decode_first_stage(sample)
                for j, m in enumerate(chunk):
                    imgs[m[0]] = dec[j * bsz:(j + 1) * bsz]
        return imgs

    def _encode_batched(self, x0, encode_text):
        g = self.generator
        bsz = x0.shape[0]
        c, uc = self._get_condition(encode_text, bsz)
        assert self.eta > 0                                                       # ddim.py:268
        jobs, order = {}, 0
        for _trial in range(self.n_trials):
            for enc_scale in self.encoder_unconditional_guidance_scales:
                for skip_steps in self.skip_steps:
                    sched = DDIMSchedule(self.custom_steps, self.eta, skip_steps, g.alphas_cumprod)
                    n_rec = max(0, min(sched.refine_steps, self.white_box_steps - skip_steps - 1))
                    noise = self._encode_noise(sched, n_rec, x0.shape)            # drawn in the reference's member order
                    jobs.setdefault((skip_steps, n_rec), []).append((order, float(enc_scale), noise))
                    order += 1
        z_ensemble = [None] * order
        for (skip_steps, n_rec), members in jobs.items():
            sched = DDIMSchedule(self.custom_steps, self.eta, skip_steps, g.alphas_cumprod)
            for chunk in self._chunks(members, bsz):
                rep = len(chunk)
                sc = torch.tensor([m[1] for m in chunk for _ in range(bsz)])
                nz = torch.cat([m[2] for m in chunk], dim=1)
                z = g.unet.latent_encode_ens(x0.repeat(rep, 1, 1, 1), c.repeat(rep, 1, 1), uc.repeat(rep, 1, 1), sc, sched, n_rec, nz)
                for j, m in enumerate(chunk):
                    z_ensemble[m[0]] = z[j * bsz:(j + 1) * bsz].reshape(bsz, -1)
        return z_ensemble

    def generate(self, z_ensemble, decode_text):
        g = self.generator
        if self.ensemble_batch and len(z_ensemble) * len(self.decoder_unconditional_guidance_scales) > 1:
            return self._generate_batched(z_ensemble, decode_text)
        img_ensemble = []
        for i, z in enumerate(z_ensemble):
            skip_steps = self.skip_steps[i % len(self.skip_steps)]
            bsz = z.shape[0]
            if self.white_box_steps != -1:
                eps_list = z.view(bsz, (self.white_box_steps - skip_steps), g.channels, g.image_size, g.image_size)
            else:
                eps_list = z.view(bsz, 1, g.channels, g.image_size, g.image_size)
            for scale in self.decoder_unconditional_guidance_scales:
                c, uc = self._get_condition(decode_text, bsz)
                sched = DDIMSchedule(self.custom_steps, self.eta, skip_steps, g.alphas_cumprod)
                n_extra = sched.refine_steps - (eps_list.shape[1] - 1)
                extra = None
                if n_extra > 0:                                                   # ddim.py:640: fresh noise where none was recovered
                    extra = torch.stack([torch.randn(eps_list[:, 0].shape) for _ in range(n_extra)])
                sample = g.unet.latent_decode(eps_list, c, uc, scale, sched, extra)
                img_ensemble.append(g.decode_first_stage(sample))
        return img_ensemble

    def encode(self, image, encode_text):
        g, e = self.generator, self.engine
        image = e.shift_scale(image, -0.5, 2.0)                                   # (image - 0.5) * 2.0
        assert image.shape[2] == image.shape[3] == self.resolution
        x0 = g.get_first_stage_encoding(g.encode_first_stage(image))
        bsz = image.shape[0]
        if self.ensemble_batch and self.n_trials * len(self.encoder_unconditional_guidance_scales) * len(self.skip_steps) > 1:
            return self._encode_batched(x0, encode_text)
        z_ensemble = []
        for _trial in range(self.n_trials):
            for enc_scale in self.encoder_unconditional_guidance_scales:
                for skip_steps in self.skip_steps:
                    c, uc = self._get_condition(encode_text, bsz)
                    assert self.eta > 0                                           # ddim.py:268
                    sched = DDIMSchedule(self.custom_steps, self.eta, skip_steps, g.alphas_cumprod)
                    n_rec = max(0, min(sched.refine_steps, self.white_box_steps - skip_steps - 1))
                    noise = self._encode_noise(sched, n_rec, x0.shape)
                    z = g.unet.latent_encode(x0, c, uc, enc_scale, sched, n_rec, noise)
                    z_ensemble.append(z.view(bsz, -1))
        return z_ensemble

    def single_member(self):
        """True when the ensemble has exactly one member whose every step is recovered (the plain CycleDiffusion cycle)."""
        if not (self.n_trials == 1 and len(self.skip_steps) == 1 and len(self.encoder_unconditional_guidance_scales) == 1
                and len(self.decoder_unconditional_guidance_scales) == 1):
            return False
        sched = DDIMSchedule(self.custom_steps, self.eta, self.skip_steps[0], self.generator.alphas_cumprod)
        return self.white_box_steps != -1 and self.white_box_steps - self.skip_steps[0] - 1 >= sched.refine_steps

    def cycle(self, image, encode_text, decode_text):
        """encode(image, encode_text) followed by forward(z, image, encode_text, decode_text) for a single-member ensemble, on the
        engine's lock-step driver (cdx_cycle_lockstep): both chains advance together, one U-Net call per step on the batch
        [source | target uncond | target cond], and the noise recovered at a step is consumed by the target chain at once -- the
        ``z`` tensor of SDW:169-206 is never materialised.  Same random draws in the same order as encode(); same result per sample
        as the two calls (tests/test_cycle_gpu.py).  Called by TextUnsupervisedTranslation.forward when single_member()."""
        assert self.single_member(), 'cycle(): single-member ensembles only (use encode() + forward())'
        g, e = self.generator, self.engine
        x = e.shift_scale(image, -0.5, 2.0)
        assert x.shape[2] == x.shape[3] == self.resolution
        x0 = g.get_first_stage_encoding(g.encode_first_stage(x))
        bsz = x.shape[0]
        c_src, uc = self._get_condition(encode_text, bsz)
        c_tgt, _ = self._get_condition(decode_text, bsz)
        assert self.eta > 0
        sched = DDIMSchedule(self.custom_steps, self.eta, self.skip_steps[0], g.alphas_cumprod)
        noise = self._encode_noise(sched, sched.refine_steps, x0.shape)
        sample = g.unet.cycle_lockstep(x0, c_src, c_tgt, uc, self.encoder_unconditional_guidance_scales[0],
                                       self.decoder_unconditional_guidance_scales[0], sched, noise)
        return e.shift_scale(g.decode_first_stage(sample), 1.0, 0.5)

    def forward(self, z_ensemble, original_img, encode_text, decode_text):
        img_ensemble = self.generate(z_ensemble, decode_text)
        assert len(img_ensemble) == len(self.decoder_unconditional_guidance_scales) * len(
            self.encoder_unconditional_guidance_scales) * len(self.skip_steps) * self.n_trials
        img_ensemble = [self.engine.shift_scale(img, 1.0, 0.5) for img in img_ensemble]     # Normalize(mean=-1, std=2)
        if len(img_ensemble) == 1:
            return img_ensemble[0]
        if self.directional_clip is None:
            raise NotImplementedError('ranking an ensemble needs ranker=<callable(img, original_img, encode_text, decode_text) -> (_, score[B])>, '
                                      'e.g. cycle_diffusion_b200.clip_rank.DirectionalCLIP(engine, clip_state_dict, tokenizer) (SURVEY.md 8f-3)')
        if hasattr(self.directional_clip, 'rank'):        # in-engine DirectionalCLIP (clip_rank.py): scores, argmax and gather stay on the device
            return self.directional_clip.rank(img_ensemble, original_img, encode_text, decode_text)[0]
        scores = []
        for img in img_ensemble:
            _, s = self.directional_clip(img, original_img, encode_text, decode_text)
            assert s.shape == (img.shape[0],)
            scores.append(s)
        best_idx = torch.argmax(torch.stack(scores, dim=1), dim=1)
        return torch.stack([img_ensemble[best_idx[b].item()][b] for b in range(best_idx.shape[0])], dim=0)

    @property
    def device(self):
        return self.engine.device


class SDStochasticTextWrapper(_StochasticTextWrapperBase):
    """Stable Diffusion v1 (512 px, latent 64, CLIP context 768, posterior *sample*)."""


class LatentDiffStochasticTextWrapper(_StochasticTextWrapperBase):
    """LDM text2img-large (256 px, latent 32, BERT context 1280, posterior *mean*: latentdiff/.../ddpm.py:537-538)."""
    RESOLUTION = 256
    LATENT = 32
    CONTEXT_DIM = 1280
    SAMPLE_POSTERIOR = False
    CKPT_DIR = 'ckpts/ldm_models'
    COND_PREFIX = 'cond_stage_model.'                 # BERTEmbedder (encoders/modules.py:79-98)
    COND_CLASS = BertTextCondStage

    @classmethod
    def default_checkpoint(cls, source_model_type):
        """LDW:21-23: ``ckpts/ldm_models/<source_model_type>/model.ckpt``."""
        return os.path.join(cls.CKPT_DIR, str(source_model_type), 'model.ckpt')


class LatentDiffStochasticWrapper(torch.nn.Module):
    """Unconditional latent-diffusion models (ffhq256 -> celeba256; VQ-f4 first stage, U-Net without context), SURVEY 8f-4.

    ref model/gan_wrapper/latentdiff_stochastic_wrapper.py:185-316: ``encode(image, class_label=None) -> z [B, white_box_steps*C*h*w]``,
    ``forward(z, class_label=None) -> img in [0,1]``, optional eta = 1 refinement pass after the decode (convsample_ddim :57-79 ->
    DDIMSampler.refine, ddim.py:114-168, 339-393).  The class-conditional branch (enforce_class_input: ClassEmbedder cross-attention
    conditioning, cin256) is not built."""

    @staticmethod
    def default_checkpoint(source_model_type):
        """latentdiff_stochastic_wrapper.py:16: ``ckpts/ldm_models/ldm/<source_model_type>/model.ckpt``."""
        return os.path.join('ckpts', 'ldm_models', 'ldm', str(source_model_type), 'model.ckpt')

    def __init__(self, source_model_type, custom_steps, eta, white_box_steps, refine_steps=0, enforce_class_input=None,
                 unconditional_guidance_scale=None, *, engine=None, device=0, state_dict=None, unet_config=None, vae_config=None,
                 latent_size=64, resolution=256, generator=None, seed=1234, alphas_cumprod=None, scale_factor=1.0):
        super().__init__()
        if enforce_class_input:
            raise NotImplementedError('class-conditional latent diffusion (ClassEmbedder conditioning) is not built; unconditional models only')
        self.enforce_class_input = enforce_class_input
        self.unconditional_guidance_scale = unconditional_guidance_scale
        self.refine_steps = refine_steps
        self.eta, self.custom_steps, self.white_box_steps = eta, custom_steps, white_box_steps
        self.vanilla = False
        if generator is not None:
            self.generator, self.engine = generator, generator.engine
        else:
            self.engine = engine or Engine(device)
            ucfg, vcfg = unet_config or specs.ldm_uncond_unet_config(), vae_config or specs.vq_f4_config()
            unet, vae = UNet(self.engine, ucfg, 'openai'), VAE(self.engine, vcfg)
            if state_dict == 'synthetic':
                unet.load_state_dict(specs.synth_state_dict(specs.openai_unet_params(ucfg), seed))
                vae.load_state_dict(specs.synth_state_dict(specs.kl_vae_params(vcfg), seed + 1))
            else:
                sd = _load_sd(state_dict, self.default_checkpoint(source_model_type), None, seed)
                unet.load_state_dict(sd, prefix='model.diffusion_model.', strict=False)
                vae.load_state_dict(sd, prefix='first_stage_model.', strict=False)
            self.generator = _LatentGenerator(self.engine, unet, vae, None, ucfg['in_channels'], latent_size, scale_factor, False)
            # ffhq256 / celeba256 LDMs: linear_start 0.0015, linear_end 0.0195 (upstream config.yaml; pass alphas_cumprod to override)
            from .schedule import ldm_alphas_cumprod
            self.generator.alphas_cumprod = alphas_cumprod if alphas_cumprod is not None else ldm_alphas_cumprod(1000, 0.0015, 0.0195)
        self.resolution = resolution
        g = self.generator
        self.latent_dim = g.image_size ** 2 * g.channels * self.white_box_steps
        self._dummy = torch.nn.Parameter(torch.zeros(1, device=self.engine.device), requires_grad=False)

    def _sched(self):
        return DDIMSchedule(self.custom_steps, self.eta, 0, self.generator.alphas_cumprod)

    def generate(self, z, class_label):
        g = self.generator
        bsz = z.shape[0]
        eps_list = z.view(bsz, self.white_box_steps, g.channels, g.image_size, g.image_size)
        sched = self._sched()
        n_extra = sched.refine_steps - (eps_list.shape[1] - 1)
        extra = torch.stack([torch.randn(eps_list[:, 0].shape) for _ in range(n_extra)]) if n_extra > 0 else None      # ddim.py:640
        sample = g.unet.latent_decode(eps_list, None, None, 1.0, sched, extra)
        return self._refine_and_decode(sample)

    def _refine_and_decode(self, sample):
        g = self.generator
        if self.refine_steps > 0:                                     # refine_eta = 1 (latentdiff_stochastic_wrapper.py:68-77)
            noise = torch.stack([torch.randn(sample.shape) for _ in range(self.refine_steps + 1)])
            sample = g.unet.latent_refine(sample, None, None, 1.0, self.custom_steps, self.refine_steps, noise, g.alphas_cumprod)
        return g.decode_first_stage(sample)

    @staticmethod
    def _encode_noise(sched, n_rec, shape):
        noise = torch.zeros((n_rec + 1,) + tuple(shape))
        noise[0] = torch.randn(shape)
        for i in range(n_rec):
            if sched.refine_steps - 1 - i != 0:                        # ddim.py:583-584: the last step returns x0 without a draw
                noise[1 + i] = torch.randn(shape)
        return noise

    def encode(self, image, class_label=None):
        g, e = self.generator, self.engine
        bsz = image.shape[0]
        image = e.shift_scale(image, -0.5, 2.0)
        assert image.shape[2] == image.shape[3] == self.resolution
        x0 = g.get_first_stage_encoding(g.encode_first_stage(image))
        assert self.eta > 0
        sched = self._sched()
        n_rec = max(0, min(sched.refine_steps, self.white_box_steps - 1))
        noise = self._encode_noise(sched, n_rec, x0.shape)
        z = g.unet.latent_encode(x0, None, None, 1.0, sched, n_rec, noise).view(bsz, -1)
        assert z.shape[1] == self.latent_dim
        return z

    def forward(self, z, class_label=None):
        return self.engine.shift_scale(self.generate(z, class_label), 1.0, 0.5)

    def pair_cycle_applies(self, target):
        """True when pair_cycle(target, image) computes target(self.encode(image)): the same DDIM schedule (custom_steps, eta,
        alphas_cumprod) and white_box_steps on both sides, the same resolution and latent shape, no class input, both models on
        one device, and every step's noise recovered by the encode (white_box_steps - 1 >= the number of DDIM steps)."""
        if not isinstance(target, LatentDiffStochasticWrapper) or self.enforce_class_input or target.enforce_class_input:
            return False
        g, h = self.generator, target.generator
        return (self.custom_steps == target.custom_steps and self.eta == target.eta and self.white_box_steps == target.white_box_steps
                and torch.equal(g.alphas_cumprod.float().cpu(), h.alphas_cumprod.float().cpu())
                and self.resolution == target.resolution and (g.channels, g.image_size) == (h.channels, h.image_size)
                and self.engine.device == target.engine.device and self.white_box_steps - 1 >= self._sched().refine_steps)

    def pair_cycle(self, target, image):
        """self.encode(image) followed by target(z), with both DDIM chains advanced in one lock-step loop (cdx_cycle_lockstep_pair:
        this model's U-Net on the source chain, the target's on the target chain, the recovered noise consumed at once -- no z
        tensor).  Same random draws in the same order as the two calls (the encode's, then the target's refinement), same result
        bit for bit.  Called by UnsupervisedTranslation.forward when pair_cycle_applies(target)."""
        assert self.pair_cycle_applies(target), 'pair_cycle(): schedules / shapes differ (use encode() + target())'
        g, e = self.generator, self.engine
        x = e.shift_scale(image, -0.5, 2.0)
        assert x.shape[2] == x.shape[3] == self.resolution
        x0 = g.get_first_stage_encoding(g.encode_first_stage(x))
        assert self.eta > 0
        sched = self._sched()
        noise = self._encode_noise(sched, sched.refine_steps, x0.shape)
        sample = g.unet.cycle_lockstep_pair(target.generator.unet, x0, None, None, None, 1.0, 1.0, sched, noise)
        return target.engine.shift_scale(target._refine_and_decode(sample), 1.0, 0.5)

    @property
    def device(self):
        return self.engine.device


class DDPMDDIMWrapper(torch.nn.Module):
    """Pixel-space DPM-Encoder / decoder (improved-DDPM U-Net for AFHQ / FFHQ)."""

    def __init__(self, source_model_type, sample_type, custom_steps, es_steps, source_model_path=None, refine_steps=0,
                 refine_iterations=1, eta=None, t_0=None, enforce_class_input=None, *, engine=None, device=0, state_dict=None,
                 image_size=None, unet=None, seed=4321, dataset=None, var_type='fixedsmall', rng='cpu'):
        super().__init__()
        # DW:360-369: the model family follows config.data.dataset -- CelebA_HQ / LSUN checkpoints are Ho et al. DDPM U-Nets
        # (models/ddpm/diffusion.py), AFHQ / FFHQ ones improved-DDPM U-Nets.  `dataset` (or a source_model_type that names one) selects it.
        # rng='cpu': every draw comes from the torch CPU generator in the reference's order (reproduces the reference CPU path under a
        # seed); rng='cuda': drawn on the engine's device (the reference's own GPU runs do this; avoids es_steps x image of host randn +
        # H2D per batch -- 1.5 GB at 250 steps, batch 8, 256^2)
        assert rng in ('cpu', 'cuda')
        self.rng = rng
        name = (dataset or str(source_model_type)).lower()
        self.model_family = 'ddpm' if any(k in name for k in ('celeba', 'lsun', 'bedroom', 'church')) else 'iddpm'
        self.enforce_class_input = enforce_class_input
        self.custom_steps, self.refine_steps, self.refine_iterations = custom_steps, refine_steps, refine_iterations
        self.sample_type, self.eta = sample_type, eta
        self.t_0 = t_0 if t_0 is not None else 999
        self.es_steps = es_steps
        if self.sample_type == 'ddim':
            assert self.eta > 0
        elif self.sample_type == 'ddpm':
            assert self.eta is None
        else:
            raise ValueError()
        if image_size is None:
            digits = ''.join(ch for ch in str(source_model_type) if ch.isdigit())
            image_size = int(digits) if digits else 256
        self.learn_sigma = False
        if unet is not None:
            self.generator, self.engine = unet, unet.engine
        else:
            self.engine = engine or Engine(device)
            if self.model_family == 'ddpm':
                cfg = specs.ddpm_config(image_size)
                params = specs.ddpm_unet_params(cfg)
            else:
                cfg = specs.iddpm_config(image_size)
                params = specs.iddpm_unet_params(cfg)
            self.generator = UNet(self.engine, cfg, self.model_family)
            sd = _load_sd(state_dict if state_dict is not None else source_model_path, source_model_path or '', params, seed)
            self.generator.load_state_dict(sd)
        self.resolution = image_size
        self.channels = 3
        self.latent_dim = self.resolution ** 2 * self.channels * self.es_steps
        self.sched = PixelSchedule(sample_type, custom_steps, es_steps, eta, self.t_0, var_type=var_type)     # config.model.var_type, DW:362-367
        self._dummy = torch.nn.Parameter(torch.zeros(1, device=self.engine.device), requires_grad=False)

    def _randn(self, shape):
        return torch.randn(shape, device=self.engine.device) if self.rng == 'cuda' else torch.randn(shape)

    def generate(self, z, class_label):
        bsz = z.shape[0]
        eps_list = z.view(bsz, self.es_steps, self.channels, self.resolution, self.resolution)
        if self.enforce_class_input:
            assert class_label is not None
            raise NotImplementedError()
        shape = eps_list[:, 0].shape
        last = self._randn(shape).unsqueeze(0)       # denoising_step draws once more; the draw is multiplied by 0 (DU:115,131)
        x = self.generator.pixel_decode(eps_list, self.sched, last_noise=last)
        return self._refine(x)

    def _refine(self, x):
        bsz, shape = x.shape[0], x.shape
        if self.refine_steps != 0:
            assert self.refine_steps < self.custom_steps
            ref = PixelSchedule(self.sample_type, self.custom_steps, self.es_steps, 1 if self.sample_type == 'ddim' else None, self.t_0)
            pairs = self.sched.pairs[-self.refine_steps:] if self.refine_steps <= len(self.sched.pairs) else self.sched.pairs
            coefs = [ref.step_coef(i, j, 1 if self.sample_type == 'ddim' else None) for i, j in pairs]
            t_loop = [float(i) for i, _ in pairs]
            at = PixelSchedule._extract(self.sched.cumprod, self.refine_steps - 1)               # DW:436-437
            for _ in range(self.refine_iterations):
                xt = self.engine.q_sample(x, self._randn(shape), at.sqrt().item(), (1 - at).sqrt().item())
                noises = torch.stack([self._randn(shape) for _ in pairs])
                x = self.generator.pixel_decode(xt.view(bsz, 1, *shape[1:]), ref, coefs=coefs, t_loop=t_loop, last_noise=noises)
        return x

    def encode(self, image, class_label=None):
        e = self.engine
        image = e.shift_scale(image, -0.5, 2.0)
        assert image.shape[2] == image.shape[3] == self.resolution
        if self.enforce_class_input:
            assert class_label is not None
            raise NotImplementedError()
        bsz = image.shape[0]
        noise = self._encode_noise(image.shape)
        z = self.generator.pixel_encode(image, self.sched, noise).view(bsz, -1)
        assert z.shape[1] == self.latent_dim
        return z

    def _encode_noise(self, shape):
        n_rec = self.es_steps - 1
        if self.rng == 'cuda':
            return torch.randn((n_rec + 1,) + tuple(shape), device=self.engine.device)
        return torch.stack([torch.randn(shape) for _ in range(n_rec + 1)])     # sample_xt, then one per sample_xt_next

    def forward(self, z, class_label=None):
        img = self.generate(z, class_label)
        return self.engine.shift_scale(img, 1.0, 0.5)

    def pair_cycle_applies(self, target):
        """True when pair_cycle(target, image) computes target(self.encode(image)): equal PixelSchedules (sample type, eta, steps,
        betas, variances), the same resolution and channels, no class input, both models on one device."""
        return (isinstance(target, DDPMDDIMWrapper) and not self.enforce_class_input and not target.enforce_class_input
                and self.resolution == target.resolution and self.channels == target.channels
                and self.engine.device == target.engine.device and self.sched.same_as(target.sched))

    def pair_cycle(self, target, image, class_label=None):
        """self.encode(image) followed by target(z) as one lock-step loop (cdx_pixel_cycle_lockstep): per step one forward of this
        model's U-Net, one of the target's and one fused kernel; the recovered noise is consumed at once, so the z tensor
        [B, es_steps*3*R*R] is never materialised.  Random draws are those of the two calls in their order -- this wrapper's encode
        buffer, then the target's last draw and refinement draws, each with its own `rng` -- and the result is the same bit for bit.
        The target's refinement (refine_steps, refine_iterations) runs unchanged afterwards.  Called by
        UnsupervisedTranslation.forward when pair_cycle_applies(target)."""
        assert self.pair_cycle_applies(target), 'pair_cycle(): schedules / shapes differ (use encode() + target())'
        e = self.engine
        x = e.shift_scale(image, -0.5, 2.0)
        assert x.shape[2] == x.shape[3] == self.resolution
        noise = self._encode_noise(x.shape)
        last = target._randn(x.shape).unsqueeze(0)              # denoising_step draws once more; the draw is multiplied by 0 (DU:115,131)
        y = self.generator.pixel_cycle_lockstep(target.generator, x, self.sched, noise, last)
        return target.engine.shift_scale(target._refine(y), 1.0, 0.5)

    @property
    def device(self):
        return self.engine.device


def get_gan_wrapper(args, target=False, **extra):
    """Same kwarg plumbing as the reference factory: every ``[gan]`` key but ``gan_type`` becomes a kwarg;
    ``target_*`` keys are renamed ``source_*`` for the target model.  ``extra`` carries engine/state_dict/... ."""
    items = list(args.items()) if isinstance(args, dict) else list(args)
    gan_type = args['gan_type'] if isinstance(args, dict) else args.gan_type
    kwargs = {}
    for kw, arg in items:
        if kw != 'gan_type':
            if (not kw.startswith('source_')) and (not kw.startswith('target_')):
                kwargs[kw] = arg
            else:
                if target and kw.startswith('target_'):
                    kwargs['source_' + kw[len('target_'):]] = arg
                elif (not target) and kw.startswith('source_'):
                    kwargs[kw] = arg
    kwargs.update(extra)
    if gan_type == "LatentDiffStochastic":
        return LatentDiffStochasticWrapper(**kwargs)
    elif gan_type == "DDPM_DDIM":
        return DDPMDDIMWrapper(**kwargs)
    elif gan_type == "LatentDiffStochasticText":
        return LatentDiffStochasticTextWrapper(**kwargs)
    elif gan_type == "SDStochasticText":
        return SDStochasticTextWrapper(**kwargs)
    else:
        raise ValueError()
