#!/usr/bin/env python
"""Generate the committed golden fixtures by running the REAL reference modules (CPU, fp32).

Run in the build container only (``/root/reference`` is not present on the GPU box):

    python tests/golden/make_golden.py

What it does
  * imports the reference's own classes -- UNetModel / SpatialTransformer (openaimodel.py, attention.py),
    VAE Encoder / Decoder (model.py), DDIMSampler (ddim.py), i-DDPM create_model (script_util.py) and
    DDPMDDIMWrapper (ddpm_ddim_wrapper.py) -- through the three shims of SURVEY.md section 8c
    (omegaconf stub, DDIMSampler.register_buffer override, LatentDiffusion stand-in);
  * loads the synthetic state_dict from ``cycle_diffusion_b200.specs`` with ``strict=True`` (this also
    pins our parameter inventories against the reference's module trees);
  * writes inputs + reference outputs to ``tests/golden/*.npz``.
Nothing from the reference is copied into the repo; only numeric outputs are stored.
"""
import contextlib
import io
import os
import sys
import tempfile
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = '/root/reference'

from cycle_diffusion_b200 import specs  # noqa: E402

torch.set_num_threads(8)


def _shim_omegaconf():
    oc = types.ModuleType('omegaconf')
    lc = types.ModuleType('omegaconf.listconfig')

    class ListConfig(list):
        pass
    lc.ListConfig = ListConfig
    oc.listconfig = lc
    oc.ListConfig = ListConfig
    sys.modules['omegaconf'] = oc
    sys.modules['omegaconf.listconfig'] = lc


def _quiet():
    return contextlib.redirect_stdout(io.StringIO())


def save(name, **arrs):
    out = {k: (v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in arrs.items()}
    path = os.path.join(HERE, name + '.npz')
    np.savez(path, **out)
    print(f'wrote {name}.npz  ({os.path.getsize(path) / 1024:.0f} KiB)')


def sd_checksum(sd):
    """Detects drift of the synthetic-weight generator between machines / torch builds."""
    s = 0.0
    a = 0.0
    for v in sd.values():
        s += float(v.double().sum())
        a += float(v.double().abs().sum())
    return np.asarray([s, a])


# ----------------------------------------------------------------------------------------------
NARROW = dict(in_channels=4, out_channels=4, model_channels=32, attention_resolutions=(4, 2, 1), num_res_blocks=2,
              channel_mult=(1, 2, 4, 4), num_heads=2, context_dim=48)
WIDE = dict(in_channels=4, out_channels=4, model_channels=320, attention_resolutions=(1, 2), num_res_blocks=1,
            channel_mult=(1, 2), num_heads=8, context_dim=768)
VAE_SMALL = dict(ch=32, ch_mult=(1, 2, 4, 4), num_res_blocks=2, in_channels=3, out_ch=3, z_channels=4, embed_dim=4)


def build_ref_unet(cfg):
    from ldm.modules.diffusionmodules.openaimodel import UNetModel
    with _quiet():
        m = UNetModel(image_size=32, in_channels=cfg['in_channels'], out_channels=cfg['out_channels'],
                      model_channels=cfg['model_channels'], attention_resolutions=list(cfg['attention_resolutions']),
                      num_res_blocks=cfg['num_res_blocks'], channel_mult=list(cfg['channel_mult']),
                      num_heads=cfg['num_heads'], use_spatial_transformer=True, transformer_depth=1,
                      context_dim=cfg['context_dim'], use_checkpoint=False, legacy=False)
    return m.eval()


def golden_unets():
    for name, cfg, seed, B, hw in (('unet_sd_narrow', NARROW, 11, 2, 16), ('unet_sd_wide', WIDE, 12, 1, 16)):
        sd = specs.synth_state_dict(specs.openai_unet_params(cfg), seed)
        m = build_ref_unet(cfg)
        m.load_state_dict(sd, strict=True)
        g = torch.Generator().manual_seed(100 + seed)
        x = torch.randn(B, cfg['in_channels'], hw, hw, generator=g)
        ctx = torch.randn(B, 77, cfg['context_dim'], generator=g)
        t = torch.tensor([901, 21][:B], dtype=torch.long)
        with torch.no_grad():
            y = m(x, t, context=ctx)
        save(name, x=x, t=t, ctx=ctx, y=y, seed=seed, wsum=sd_checksum(sd))


def golden_vae():
    from ldm.modules.diffusionmodules.model import Encoder, Decoder
    cfg = VAE_SMALL
    sd = specs.synth_state_dict(specs.kl_vae_params(cfg), 21)
    dd = dict(double_z=True, z_channels=cfg['z_channels'], resolution=64, in_channels=3, out_ch=3, ch=cfg['ch'],
              ch_mult=list(cfg['ch_mult']), num_res_blocks=cfg['num_res_blocks'], attn_resolutions=[], dropout=0.0)
    with _quiet():
        enc, dec = Encoder(**dd).eval(), Decoder(**dd).eval()
    enc.load_state_dict({k[len('encoder.'):]: v for k, v in sd.items() if k.startswith('encoder.')}, strict=True)
    dec.load_state_dict({k[len('decoder.'):]: v for k, v in sd.items() if k.startswith('decoder.')}, strict=True)
    quant = torch.nn.Conv2d(2 * cfg['z_channels'], 2 * cfg['embed_dim'], 1)
    post = torch.nn.Conv2d(cfg['embed_dim'], cfg['z_channels'], 1)
    quant.load_state_dict({'weight': sd['quant_conv.weight'], 'bias': sd['quant_conv.bias']})
    post.load_state_dict({'weight': sd['post_quant_conv.weight'], 'bias': sd['post_quant_conv.bias']})
    g = torch.Generator().manual_seed(121)
    img = torch.rand(2, 3, 64, 64, generator=g) * 2 - 1
    z = torch.randn(2, 4, 8, 8, generator=g)
    with torch.no_grad():
        moments = quant(enc(img))           # AutoencoderKL.encode, autoencoder.py:324-328
        rec = dec(post(z))                  # AutoencoderKL.decode, autoencoder.py:330-333
    save('vae_small', img=img, z=z, moments=moments, rec=rec, seed=21, wsum=sd_checksum(sd))


def golden_iddpm():
    sys.path.insert(0, os.path.join(REF, 'model/lib/ddpm_ddim'))
    from models.improved_ddpm.script_util import create_model, AFHQ_DICT
    cfg = specs.iddpm_config(64)
    sd = specs.synth_state_dict(specs.iddpm_unet_params(cfg), 31)
    with _quiet():
        m = create_model(**{**AFHQ_DICT, 'image_size': 64}).eval()
    m.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(131)
    x = torch.randn(2, 3, 64, 64, generator=g)
    t = torch.tensor([500., 3.])
    with torch.no_grad():
        y = m(x, t)
    save('unet_iddpm64', x=x, t=t, y=y, seed=31, wsum=sd_checksum(sd))
    # also pin the 256 inventory (no forward: just strict key/shape check)
    cfg256 = specs.iddpm_config(256)
    with _quiet():
        m256 = create_model(**AFHQ_DICT)
    ref_keys = {k: tuple(v.shape) for k, v in m256.state_dict().items()}
    ours = {k: tuple(s) for k, s, _ in specs.iddpm_unet_params(cfg256)}
    assert ref_keys == ours, 'i-DDPM 256 inventory mismatch'
    print('i-DDPM 256 inventory matches the reference module tree')


def golden_inventories():
    """Full-size SD / LDM U-Net and KL-f8 VAE inventories against the reference module trees (meta device)."""
    from ldm.modules.diffusionmodules.openaimodel import UNetModel
    from ldm.modules.diffusionmodules.model import Encoder, Decoder
    for ctx in (768, 1280):
        cfg = specs.sd_unet_config(ctx)
        with torch.device('meta'), _quiet():
            m = UNetModel(image_size=32, in_channels=4, out_channels=4, model_channels=320,
                          attention_resolutions=[4, 2, 1], num_res_blocks=2, channel_mult=[1, 2, 4, 4], num_heads=8,
                          use_spatial_transformer=True, transformer_depth=1, context_dim=ctx, use_checkpoint=True,
                          legacy=False)
        ref = {k: tuple(v.shape) for k, v in m.state_dict().items()}
        ours = {k: tuple(s) for k, s, _ in specs.openai_unet_params(cfg)}
        assert ref == ours, f'SD U-Net inventory mismatch (ctx {ctx})'
    cfg = specs.kl_f8_config()
    dd = dict(double_z=True, z_channels=4, resolution=256, in_channels=3, out_ch=3, ch=128, ch_mult=[1, 2, 4, 4],
              num_res_blocks=2, attn_resolutions=[], dropout=0.0)
    with torch.device('meta'), _quiet():
        enc, dec = Encoder(**dd), Decoder(**dd)
    ref = {'encoder.' + k: tuple(v.shape) for k, v in enc.state_dict().items()}
    ref.update({'decoder.' + k: tuple(v.shape) for k, v in dec.state_dict().items()})
    ours = {k: tuple(s) for k, s, _ in specs.kl_vae_params(cfg) if not k.startswith(('quant', 'post_quant'))}
    assert ref == ours, 'KL-f8 inventory mismatch'
    print('SD/LDM U-Net and KL-f8 VAE inventories match the reference module trees')


# ----------------------------------------------------------------------------------------------
def golden_schedule():
    from ldm.modules.diffusionmodules.util import make_beta_schedule, make_ddim_timesteps, make_ddim_sampling_parameters
    betas = make_beta_schedule('linear', 1000, linear_start=0.00085, linear_end=0.012)
    ac = torch.tensor(np.cumprod(1. - betas, axis=0), dtype=torch.float32)   # register_schedule, ddpm.py:124-135
    out = {'alphas_cumprod': ac}
    for S in (10, 50, 99, 100):
        ts = make_ddim_timesteps('uniform', S, 1000, verbose=False)
        sig, a, ap = make_ddim_sampling_parameters(ac.cpu(), ts, 0.1, verbose=False)
        # what the step functions finally consume: torch.full((b,1,1,1), table[index]) -> fp32
        f32 = lambda tab: torch.stack([torch.full((1,), tab[i]) for i in range(S)]).flatten()
        out[f'ts_{S}'] = ts
        out[f'a_{S}'] = f32(a)
        out[f'aprev_{S}'] = f32(ap)
        out[f'sigma_{S}'] = f32(sig)
        out[f'sqrt1ma_{S}'] = f32(np.sqrt(1. - a))
    save('schedule_ldm', **out)


class _LatentStandIn:
    """What DDIMSampler touches on ``self.model`` (ddpm.py:117-145, 882-983, 1386-1394)."""

    def __init__(self, unet):
        from ldm.modules.diffusionmodules.util import make_beta_schedule
        betas = make_beta_schedule('linear', 1000, linear_start=0.00085, linear_end=0.012)
        ac = np.cumprod(1. - betas, axis=0)
        self.num_timesteps = 1000
        self.betas = torch.tensor(betas, dtype=torch.float32)
        self.alphas_cumprod = torch.tensor(ac, dtype=torch.float32)
        self.alphas_cumprod_prev = torch.tensor(np.append(1., ac[:-1]), dtype=torch.float32)
        self.device = torch.device('cpu')
        self.parameterization = 'eps'
        self.unet = unet

    def apply_model(self, x, t, c):
        return self.unet(x, t, context=c)


def golden_ddim_cycle():
    from ldm.models.diffusion.ddim import DDIMSampler

    class CPUSampler(DDIMSampler):
        def register_buffer(self, name, attr):      # stock one forces .to("cuda"), ddim.py:19-23
            setattr(self, name, attr)

    cfg = NARROW
    sd = specs.synth_state_dict(specs.openai_unet_params(cfg), 11)
    unet = build_ref_unet(cfg)
    unet.load_state_dict(sd, strict=True)
    model = _LatentStandIn(unet)
    g = torch.Generator().manual_seed(141)
    B = 2
    x0 = torch.randn(B, 4, 16, 16, generator=g) * 0.8
    c_src = torch.randn(B, 77, 48, generator=g)
    c_tgt = torch.randn(B, 77, 48, generator=g)
    uc = torch.randn(B, 77, 48, generator=g)
    out = dict(x0=x0, c_src=c_src, c_tgt=c_tgt, uc=uc)
    for tag, S, skip, wb, enc_scale, dec_scale in (('a', 10, 3, 11, 1.0, 3.0), ('b', 8, 0, 9, 2.0, 1.0)):
        torch.manual_seed(1000 + S)
        with torch.no_grad(), _quiet():
            z_list = CPUSampler(model).ddpm_ddim_encoding(S, conditioning=c_src, batch_size=B, shape=(4, 16, 16), eta=0.1,
                                                          white_box_steps=wb, skip_steps=skip, verbose=False, x0=x0,
                                                          unconditional_guidance_scale=enc_scale,
                                                          unconditional_conditioning=uc)
            z = torch.stack(z_list, dim=1).view(B, -1)                       # SDW:203
            eps_list = z.view(B, wb - skip, 4, 16, 16)                         # SDW:150
            x_T, eps = eps_list[:, 0], eps_list[:, 1:]
            same, _ = CPUSampler(model).sample_with_eps(S, eps, conditioning=c_src, batch_size=B, shape=(4, 16, 16),
                                                        eta=0.1, verbose=False, x_T=x_T, skip_steps=skip,
                                                        unconditional_guidance_scale=enc_scale,
                                                        unconditional_conditioning=uc)
            tgt, _ = CPUSampler(model).sample_with_eps(S, eps, conditioning=c_tgt, batch_size=B, shape=(4, 16, 16),
                                                       eta=0.1, verbose=False, x_T=x_T, skip_steps=skip,
                                                       unconditional_guidance_scale=dec_scale,
                                                       unconditional_conditioning=uc)
        print(f'ddim_cycle[{tag}]: same-condition reconstruction max|x0_hat-x0| = {(same - x0).abs().max():.3e}, '
              f'|z|max = {z.abs().max():.2f}')
        out.update({f'z_{tag}': z, f'same_{tag}': same, f'tgt_{tag}': tgt,
                    f'cfg_{tag}': np.asarray([S, skip, wb, enc_scale, dec_scale, 1000 + S], dtype=np.float64)})
    save('ddim_cycle_narrow', **out)


def golden_pixel_cycle():
    """cfg1: DDPMDDIMWrapper as-is on a 64x64 i-DDPM U-Net, 10 encode + 10 decode steps, B=1, plus a ddpm-type run."""
    cfg = specs.iddpm_config(64)
    sd = specs.synth_state_dict(specs.iddpm_unet_params(cfg), 31)
    cwd = os.getcwd()
    tmp = tempfile.mkdtemp()
    os.makedirs(os.path.join(tmp, 'ckpts/ddpm/configs'))
    with open(os.path.join(tmp, 'ckpts/ddpm/configs/afhq.yml'), 'w') as f:
        f.write('data:\n  dataset: AFHQ\n  image_size: 64\n  channels: 3\n'
                'diffusion:\n  beta_start: 0.0001\n  beta_end: 0.02\n  num_diffusion_timesteps: 1000\n')
    torch.save(sd, os.path.join(tmp, 'ckpts/ddpm/afhq64.pt'))
    sys.path.insert(0, REF)
    os.chdir(tmp)
    try:
        with _quiet():
            import model.gan_wrapper.ddpm_ddim_wrapper as W
        from model.lib.ddpm_ddim.models.improved_ddpm.script_util import create_model, AFHQ_DICT
        W.i_DDPM = lambda name='AFHQ': create_model(**{**AFHQ_DICT, 'image_size': 64})
        out = {}
        g = torch.Generator().manual_seed(151)
        image = torch.rand(1, 3, 64, 64, generator=g)
        out['image'] = image
        for tag, kw in (('ddim', dict(sample_type='ddim', eta=0.1, custom_steps=10, es_steps=10)),
                        ('ddpm', dict(sample_type='ddpm', eta=None, custom_steps=20, es_steps=6)),
                        # eta=1 refinement after the decode (DW:431-453): 3 steps, 2 iterations, fresh noise each
                        ('ddim_refine', dict(sample_type='ddim', eta=0.1, custom_steps=10, es_steps=10, refine_steps=3, refine_iterations=2))):
            kw = dict(kw)
            kw.setdefault('refine_steps', 0)
            with _quiet():
                w = W.DDPMDDIMWrapper(source_model_type='afhqcat256', source_model_path='ckpts/ddpm/afhq64.pt', **kw)
            torch.manual_seed(2000)
            with torch.no_grad(), _quiet():
                z = w.encode(image)
                st = torch.get_rng_state()
                img = w(z)
                # conditioning of the decode map: the reference's own output change for a 1-ulp relative change of z
                # under identical noise draws (the GPU tests scale their tolerance with it)
                torch.set_rng_state(st)
                img_p = w(z * (1 + 2.0 ** -23))
            out[f'z_{tag}'] = z
            out[f'img_{tag}'] = img
            out[f'sens_{tag}'] = (img_p - img).abs().max().reshape(1)
            print(f'pixel_cycle[{tag}]: 1-ulp sensitivity of the reference decode {float(out[f"sens_{tag}"]):.3e}')
            print(f'pixel_cycle[{tag}]: z {tuple(z.shape)} |z|max {z.abs().max():.2f}  recon max|img-image| '
                  f'{(img - image).abs().max():.3e}')
        # the refinement acts on the decode only: its z is the 'ddim' encode, stored once (keeps the fixture under 1 MB)
        assert torch.equal(out.pop('z_ddim_refine'), out['z_ddim'])
        save('pixel_cycle_iddpm64', **out)
    finally:
        os.chdir(cwd)


def golden_clip_text():
    """CLIP text tower: the installed transformers CLIPTextModel (the third-party model FrozenCLIPEmbedder wraps,
    encoders/modules.py:140-158) on two reduced configs with our synthetic weights loaded strict=True."""
    from transformers import CLIPTextConfig, CLIPTextModel
    out = {}
    for tag, c in (('small', specs.clip_text_config(vocab_size=1000, width=64, layers=2, heads=4, max_len=77, mlp_width=256)),
                   ('wide', specs.clip_text_config(vocab_size=2000, width=128, layers=3, heads=2, max_len=77, mlp_width=512))):
        hf = CLIPTextConfig(vocab_size=c['vocab_size'], hidden_size=c['width'], intermediate_size=c['mlp_width'],
                            num_hidden_layers=c['layers'], num_attention_heads=c['heads'], max_position_embeddings=c['max_len'],
                            hidden_act='quick_gelu', layer_norm_eps=1e-5)
        m = CLIPTextModel(hf).eval()
        sd = specs.synth_state_dict(specs.clip_text_params(c), 77 + c['width'], gain=2.0)
        want = {k for k in m.state_dict() if not k.endswith('position_ids')}
        assert want == set(sd), (sorted(want ^ set(sd))[:6])
        m.load_state_dict(sd, strict=False)
        g = torch.Generator().manual_seed(5 + c['width'])
        ids = torch.randint(0, c['vocab_size'], (3, 77), generator=g)
        ids_short = ids[:2, :19].contiguous()
        with torch.no_grad():
            y = m(input_ids=ids).last_hidden_state
            ys = m(input_ids=ids_short).last_hidden_state
        out.update({f'ids_{tag}': ids, f'out_{tag}': y, f'ids_short_{tag}': ids_short, f'out_short_{tag}': ys,
                    f'cfg_{tag}': np.asarray([c[k] for k in ('vocab_size', 'width', 'layers', 'heads', 'max_len', 'mlp_width')], dtype=np.int64)})
        print(f'clip_text[{tag}]: out {tuple(y.shape)} |y|max {y.abs().max():.3f}')
    save('clip_text', **out)


def golden_bert_text():
    """LDM BERTEmbedder: the reference's own x_transformer TransformerWrapper(Encoder(dim, depth)) exactly as
    encoders/modules.py:88-90 builds it (the module file itself imports clip/kornia, so its three lines are restated here)."""
    from ldm.modules.x_transformer import Encoder, TransformerWrapper
    out = {}
    for tag, c in (('small', specs.bert_text_config(vocab_size=500, width=96, layers=2)),
                   ('wide', specs.bert_text_config(vocab_size=800, width=256, layers=3))):
        m = TransformerWrapper(num_tokens=c['vocab_size'], max_seq_len=c['max_len'], attn_layers=Encoder(dim=c['width'], depth=c['layers']),
                               emb_dropout=0.0).eval()
        sd = specs.synth_state_dict(specs.bert_text_params(c), 11 + c['width'], gain=2.0)
        want = {k[len('transformer.'):] for k in sd}
        have = {k for k in m.state_dict() if not k.startswith('to_logits.')}
        assert want == have, sorted(want ^ have)[:6]
        m.load_state_dict({k[len('transformer.'):]: v for k, v in sd.items()}, strict=False)
        g = torch.Generator().manual_seed(9 + c['width'])
        tok = torch.randint(0, c['vocab_size'], (3, 77), generator=g)
        with torch.no_grad():
            y = m(tok, return_embeddings=True)
        out.update({f'tok_{tag}': tok, f'out_{tag}': y,
                    f'cfg_{tag}': np.asarray([c[k] for k in ('vocab_size', 'width', 'layers', 'heads', 'dim_head', 'max_len', 'mlp_width')], dtype=np.int64)})
        print(f'bert_text[{tag}]: out {tuple(y.shape)} |y|max {y.abs().max():.3f}')
    save('bert_text', **out)


def golden_clip_rank():
    """Directional-CLIP ranking (SURVEY 8f-3).  Features / scores: the installed transformers CLIPModel (the HF restatement of the
    OpenAI CLIP model clean_clip.py:10 loads) on a reduced ViT config with synthetic weights loaded strict; preprocessing as the
    reference's tensor path (bicubic, no antialias).  Metrics: the reference's OWN evaluation/utils.py functions."""
    from transformers import CLIPConfig, CLIPModel, CLIPTextConfig, CLIPVisionConfig
    import torch.nn.functional as F
    vc = dict(kind='clip_vision', width=64, layers=2, heads=4, mlp_width=256, patch=8, image_size=32, proj_dim=48)
    tc = dict(kind='clip', vocab_size=600, width=96, layers=2, heads=4, max_len=77, mlp_width=384, proj_dim=48)
    cfg = CLIPConfig(text_config=CLIPTextConfig(vocab_size=tc['vocab_size'], hidden_size=tc['width'], intermediate_size=tc['mlp_width'],
                                                num_hidden_layers=tc['layers'], num_attention_heads=tc['heads'], max_position_embeddings=77,
                                                hidden_act='quick_gelu', layer_norm_eps=1e-5, projection_dim=48, eos_token_id=2).to_dict(),
                     vision_config=CLIPVisionConfig(hidden_size=vc['width'], intermediate_size=vc['mlp_width'], num_hidden_layers=vc['layers'],
                                                    num_attention_heads=vc['heads'], image_size=32, patch_size=8, hidden_act='quick_gelu',
                                                    layer_norm_eps=1e-5, projection_dim=48).to_dict(), projection_dim=48)
    m = CLIPModel(cfg).eval()
    sd = dict(specs.synth_state_dict(specs.clip_vision_params(vc), 31, gain=2.0))
    sd.update(specs.synth_state_dict(specs.clip_text_params(tc) + [('text_projection.weight', (48, tc['width']), 'w')], 32, gain=2.0))
    want = {k for k in m.state_dict() if not k.endswith('position_ids') and k != 'logit_scale'}
    assert want == set(sd), sorted(want ^ set(sd))[:8]
    m.load_state_dict(sd, strict=False)
    g = torch.Generator().manual_seed(17)
    img, orig = torch.rand(3, 3, 80, 80, generator=g), torch.rand(3, 3, 80, 80, generator=g)
    ids_e, ids_d = torch.randint(3, 599, (3, 77), generator=g), torch.randint(3, 599, (3, 77), generator=g)
    for t in (ids_e, ids_d):                     # CLIP tokenisation: the EOT token has the LARGEST id and sits at a different place per prompt
        for b, pos in enumerate((5, 19, 76)):
            t[b, pos] = 599
    mean = torch.tensor([0.48145466, 0.4578275, 0.40821073]).view(1, 3, 1, 1)
    std = torch.tensor([0.26862954, 0.26130258, 0.27577711]).view(1, 3, 1, 1)
    pre = lambda x: (F.interpolate(x, size=(32, 32), mode='bicubic', align_corners=False) - mean) / std
    with torch.no_grad():
        pi, po = pre(img), pre(orig)
        fi = m.vision_model(pixel_values=pi).pooler_output @ m.visual_projection.weight.t()        # == get_image_features
        fo = m.vision_model(pixel_values=po).pooler_output @ m.visual_projection.weight.t()
        # (transformers pools at eos_token_id; the OpenAI model pools at argmax(ids) -- same position here by construction)
        te = m.text_model(input_ids=ids_e).last_hidden_state[torch.arange(3), ids_e.argmax(-1)] @ m.text_projection.weight.t()
        td = m.text_model(input_ids=ids_d).last_hidden_state[torch.arange(3), ids_d.argmax(-1)] @ m.text_projection.weight.t()
        n = lambda t: t / t.norm(dim=-1, keepdim=True)
        fi_, fo_, te_, td_ = n(fi), n(fo), n(te), n(td)
        clip = torch.einsum('bz,bz->b', fi_, td_)
        dclip = torch.einsum('bz,bz->b', n(fi_ - fo_), n(td_ - te_))
    # metrics from the reference's own functions (evaluation/utils.py; call site evaluation/translate_text.py:76-89)
    sys.path.insert(0, REF)
    from evaluation.utils import calculate_psnr, calculate_ssim
    a = (torch.rand(2, 3, 48, 40, generator=g) * 1.2 - 0.1)
    b = (a + 0.1 * torch.randn(2, 3, 48, 40, generator=g))
    met = []
    for x, y in zip(a, b):
        x, y = x.clamp(0, 1), y.clamp(0, 1)
        met.append([calculate_psnr(x, y).item(),
                    calculate_ssim((x.numpy() * 255).transpose((1, 2, 0)), (y.numpy() * 255).transpose((1, 2, 0))),
                    torch.sqrt(((x - y) ** 2).sum(2).sum(1).sum(0)).item()])
    save('clip_rank', img=img, orig=orig, ids_e=ids_e, ids_d=ids_d, pre_img=pi, f_img=fi, f_orig=fo, f_enc=te, f_dec=td, clip=clip, dclip=dclip,
         met_a=a, met_b=b, met=np.asarray(met, dtype=np.float64))
    print(f'clip_rank: clip {clip.tolist()} dclip {dclip.tolist()} metrics {met}')


UNCOND_SMALL = dict(in_channels=3, out_channels=3, model_channels=32, attention_resolutions=(2, 4), num_res_blocks=1,
                    channel_mult=(1, 2, 2), num_head_channels=16, context_dim=0)
VQ_SMALL = dict(ch=32, ch_mult=(1, 2, 4), num_res_blocks=1, in_channels=3, out_ch=3, z_channels=3, embed_dim=3, vq=True, n_embed=256)


def golden_ldm_uncond():
    """SURVEY 8f-4: the unconditional LDM path of LatentDiffStochasticWrapper.  (i) the reference UNetModel built with
    use_spatial_transformer=False (AttentionBlock + QKVAttentionLegacy); (ii) the reference VAE Encoder / Decoder with double_z=False
    around the VQ 1x1 convs, quantiser restated (taming is absent from the tree); (iii) DDIMSampler: ddpm_ddim_encoding with no
    conditioning -> sample_with_eps -> refine(eta=1), the call sequence of latentdiff_stochastic_wrapper.py:57-79, 164-170."""
    from ldm.modules.diffusionmodules.openaimodel import UNetModel
    from ldm.modules.diffusionmodules.model import Encoder, Decoder
    from ldm.models.diffusion.ddim import DDIMSampler

    class CPUSampler(DDIMSampler):
        def register_buffer(self, name, attr):
            setattr(self, name, attr)

    cfg = UNCOND_SMALL
    sd = specs.synth_state_dict(specs.openai_unet_params(cfg), 41)
    with _quiet():
        unet = UNetModel(image_size=16, in_channels=3, out_channels=3, model_channels=cfg['model_channels'],
                         attention_resolutions=list(cfg['attention_resolutions']), num_res_blocks=cfg['num_res_blocks'],
                         channel_mult=list(cfg['channel_mult']), num_head_channels=cfg['num_head_channels'], use_spatial_transformer=False,
                         use_checkpoint=False).eval()
    unet.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(241)
    x = torch.randn(2, 3, 16, 16, generator=g)
    t = torch.tensor([801, 41], dtype=torch.long)
    with torch.no_grad():
        y = unet(x, t)
    out = dict(x=x, t=t, y=y, wsum=sd_checksum(sd))
    # (ii) VQ first stage
    vc = VQ_SMALL
    vsd = specs.synth_state_dict(specs.kl_vae_params(vc), 42)
    dd = dict(double_z=False, z_channels=3, resolution=64, in_channels=3, out_ch=3, ch=vc['ch'], ch_mult=list(vc['ch_mult']),
              num_res_blocks=vc['num_res_blocks'], attn_resolutions=[], dropout=0.0)
    with _quiet():
        enc, dec = Encoder(**dd).eval(), Decoder(**dd).eval()
    enc.load_state_dict({k[len('encoder.'):]: v for k, v in vsd.items() if k.startswith('encoder.')}, strict=True)
    dec.load_state_dict({k[len('decoder.'):]: v for k, v in vsd.items() if k.startswith('decoder.')}, strict=True)
    img = torch.rand(2, 3, 64, 64, generator=g) * 2 - 1
    zz = torch.randn(2, 3, 16, 16, generator=g) * 0.5
    import torch.nn.functional as F
    with torch.no_grad():
        h = F.conv2d(enc(img), vsd['quant_conv.weight'], vsd['quant_conv.bias'])                 # VQModelInterface.encode
        emb = vsd['quantize.embedding.weight']
        zp = zz.permute(0, 2, 3, 1).contiguous()
        zf = zp.view(-1, 3)
        d = torch.sum(zf ** 2, dim=1, keepdim=True) + torch.sum(emb ** 2, dim=1) - 2 * torch.einsum('bd,dn->bn', zf, emb.t())
        zq = emb[torch.argmin(d, dim=1)].view(zp.shape)
        zq = (zp + (zq - zp)).permute(0, 3, 1, 2).contiguous()
        rec = dec(F.conv2d(zq, vsd['post_quant_conv.weight'], vsd['post_quant_conv.bias']))     # VQModelInterface.decode
    out.update(img=img, h=h, zz=zz, rec=rec)
    # (iii) sampler sequence
    model = _LatentStandIn(unet)
    model.apply_model = lambda xx, tt, cc: unet(xx, tt)
    x0 = torch.randn(2, 3, 16, 16, generator=g) * 0.7
    S, wb, r = 8, 9, 3
    torch.manual_seed(4242)
    with torch.no_grad(), _quiet():
        z_list = CPUSampler(model).ddpm_ddim_encoding(S, batch_size=2, shape=(3, 16, 16), eta=0.1, white_box_steps=wb, verbose=False, x0=x0)
        z = torch.stack(z_list, dim=1).view(2, -1)
        eps_list = z.view(2, wb, 3, 16, 16)
        dec_, _ = CPUSampler(model).sample_with_eps(S, eps_list[:, 1:], batch_size=2, shape=(3, 16, 16), eta=0.1, verbose=False, x_T=eps_list[:, 0])
        ref_, _ = CPUSampler(model).refine(S, refine_steps=r, batch_size=2, shape=(3, 16, 16), eta=1, verbose=False, x0=dec_)
    print(f'ldm_uncond: unet |y|max {y.abs().max():.3f}  cycle |dec - x0| {(dec_ - x0).abs().max():.2e}  |refined - dec| {(ref_ - dec_).abs().max():.3f}')
    out.update(x0=x0, z=z, dec=dec_, refined=ref_, cyc=np.asarray([S, wb, r, 4242], dtype=np.int64))
    save('ldm_uncond', **out)


DDPM_SMALL = dict(image_size=32, in_channels=3, out_channels=3, model_channels=32, num_res_blocks=2, channel_mult=(1, 2, 2), attention_resolutions=(2,))


def golden_unet_ddpm():
    """SURVEY 8f-4: the reference's own Ho-et-al ``DDPM`` class (models/ddpm/diffusion.py) on a reduced config, synthetic weights strict."""
    sys.path.insert(0, os.path.join(REF, 'model/lib/ddpm_ddim'))
    from models.ddpm.diffusion import DDPM
    from types import SimpleNamespace as NS
    cfg = DDPM_SMALL
    conf = NS(model=NS(ch=32, out_ch=3, ch_mult=(1, 2, 2), num_res_blocks=2, attn_resolutions=[16], dropout=0.0, in_channels=3, resamp_with_conv=True),
              data=NS(image_size=32))
    m = DDPM(conf).eval()
    sd = specs.synth_state_dict(specs.ddpm_unet_params(cfg), 61)
    assert set(m.state_dict()) == set(sd), sorted(set(m.state_dict()) ^ set(sd))[:8]
    m.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(261)
    x = torch.randn(2, 3, 32, 32, generator=g)
    t = torch.tensor([999., 3.])
    with torch.no_grad():
        y = m(x, t)
    print(f'unet_ddpm: |y|max {y.abs().max():.3f}')
    save('unet_ddpm', x=x, t=t, y=y, wsum=sd_checksum(sd))


if __name__ == '__main__':
    _shim_omegaconf()
    sys.path.insert(0, os.path.join(REF, 'model/lib/stable_diffusion'))
    golden_inventories()
    golden_schedule()
    golden_unets()
    golden_vae()
    golden_ddim_cycle()
    golden_iddpm()
    golden_pixel_cycle()
    golden_clip_text()
    golden_bert_text()
    golden_clip_rank()
    golden_ldm_uncond()
    golden_unet_ddpm()
