"""Path-level parity on the GPU: DPM-Encoder inversion + decode loops and the drop-in wrappers, against the
reference-generated fixtures and the CPU oracle under the same torch.manual_seed.

The recovered noise z is amplified by 1/sigma_t (|z| reaches 1e2-1e3 with synthetic weights), so z is compared
relative to its own max; decoded latents / images use the north-star bar |delta| <= 1e-3 (fp32 latents)."""
import pytest
import torch

from cycle_diffusion_b200 import specs
from tests.common import NARROW, VAE_SMALL, golden, maxdiff

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def eng():
    from cycle_diffusion_b200.engine import Engine
    return Engine(0)


def _encode_noise(sched, n_rec, shape):
    noise = torch.zeros((n_rec + 1,) + tuple(shape))
    noise[0] = torch.randn(shape)
    for i in range(n_rec):
        if sched.refine_steps - 1 - i != 0:
            noise[1 + i] = torch.randn(shape)
    return noise


@pytest.mark.parametrize('tag', ['a', 'b'])
def test_latent_cycle_vs_reference_fixture(eng, tag):
    from cycle_diffusion_b200.engine import UNet
    from cycle_diffusion_b200.schedule import DDIMSchedule
    g = golden('ddim_cycle_narrow')
    S, skip, wb, enc_scale, dec_scale, seed = [float(v) for v in g[f'cfg_{tag}']]
    S, skip, wb, seed = int(S), int(skip), int(wb), int(seed)
    sd = specs.synth_state_dict(specs.openai_unet_params(NARROW), 11)
    unet = UNet(eng, NARROW, 'openai').load_state_dict(sd)
    sched = DDIMSchedule(S, 0.1, skip)
    n_rec = min(sched.refine_steps, wb - skip - 1)
    torch.manual_seed(seed)
    noise = _encode_noise(sched, n_rec, g['x0'].shape)
    z = unet.latent_encode(g['x0'], g['c_src'], g['uc'], enc_scale, sched, n_rec, noise)
    zref = g[f'z_{tag}'].view(z.shape)
    rz = maxdiff(z.cpu(), zref) / float(zref.abs().max())
    same = unet.latent_decode(zref, g['c_src'], g['uc'], enc_scale, sched).cpu()
    tgt = unet.latent_decode(zref, g['c_tgt'], g['uc'], dec_scale, sched).cpu()
    own = unet.latent_decode(z, g['c_src'], g['uc'], enc_scale, sched).cpu()       # engine encode -> engine decode
    print(f'cycle[{tag}]: rel|dz| {rz:.2e}  |d same| {maxdiff(same, g[f"same_{tag}"]):.2e}  |d tgt| {maxdiff(tgt, g[f"tgt_{tag}"]):.2e}'
          f'  own-cycle |x0_hat - x0| {maxdiff(own, g["x0"]):.2e}')
    assert rz < 2e-4
    assert maxdiff(same, g[f'same_{tag}']) < 1e-3
    assert maxdiff(tgt, g[f'tgt_{tag}']) < 1e-3
    assert maxdiff(own, g['x0']) < 1e-3


@pytest.mark.parametrize('tag,kw', [('ddim', dict(sample_type='ddim', eta=0.1, custom_steps=10, es_steps=10)),
                                    ('ddpm', dict(sample_type='ddpm', eta=None, custom_steps=20, es_steps=6)),
                                    ('ddim_refine', dict(sample_type='ddim', eta=0.1, custom_steps=10, es_steps=10, refine_steps=3,
                                                         refine_iterations=2))])
def test_pixel_wrapper_vs_reference_fixture(eng, tag, kw):
    """BASELINE config 1: DDPMDDIMWrapper on the 64x64 i-DDPM U-Net, fixture from the unmodified reference wrapper."""
    from cycle_diffusion_b200.wrappers import DDPMDDIMWrapper
    g = golden('pixel_cycle_iddpm64')
    cfg = specs.iddpm_config(64)
    sd = specs.synth_state_dict(specs.iddpm_unet_params(cfg), 31)
    w = DDPMDDIMWrapper('afhqcat64', source_model_path=None, state_dict=sd, image_size=64, engine=eng, **kw)
    assert (w.resolution, w.channels, w.latent_dim) == (64, 3, 64 * 64 * 3 * kw['es_steps'])
    torch.manual_seed(2000)
    z = w.encode(g['image'])
    zref = g['z_ddim' if tag == 'ddim_refine' else f'z_{tag}']       # the refinement acts on the decode only: same encode as 'ddim'
    rz = maxdiff(z.cpu(), zref) / float(zref.abs().max())
    # (the fixture's decode continues the encode's CPU RNG stream; our encode consumed the same number of draws)
    img = w(zref).cpu()
    print(f'pixel[{tag}]: rel|dz| {rz:.2e}  |d img| {maxdiff(img, g[f"img_{tag}"]):.2e}')
    assert z.shape == zref.shape
    assert rz < 5e-4
    # tolerance: 1e-3, widened only where the reference's OWN decode is ill-conditioned: sens_* is the change of the reference
    # output for a 1-ulp relative perturbation of z under identical noise (5.5e-4 for the eta=1 refinement, whose output
    # leaves [0,1] and reaches 2.7 with synthetic weights)
    tol = max(1e-3, 8 * float(g[f'sens_{tag}']))
    assert maxdiff(img, g[f'img_{tag}']) < tol
    with pytest.raises(AssertionError):
        w.encode(torch.rand(1, 3, 32, 32))                 # DW:472 resolution check


def test_sd_wrapper_vs_oracle_end_to_end(eng):
    """SDStochasticTextWrapper surface (encode -> forward) on a small SD-topology model against the CPU oracle's
    restatement of the same wrapper, same seeds: VAE encode + posterior sample + DPM-Encoder + CFG decode + VAE decode."""
    from cycle_diffusion_b200.wrappers import SDStochasticTextWrapper, SyntheticTextEncoder
    from oracle import dpm_encoder, unet_openai, vae_kl
    usd = specs.synth_state_dict(specs.openai_unet_params(NARROW), 11)
    vsd = specs.synth_state_dict(specs.kl_vae_params(VAE_SMALL), 21)
    sd = {'model.diffusion_model.' + k: v for k, v in usd.items()}
    sd.update({'first_stage_model.' + k: v for k, v in vsd.items()})
    cond = SyntheticTextEncoder(48)
    kw = dict(custom_steps=6, eta=0.1, white_box_steps=7, skip_steps=[2], encoder_unconditional_guidance_scales=[1.0],
              decoder_unconditional_guidance_scales=[3.0], n_trials=1)
    w = SDStochasticTextWrapper('synthetic', engine=eng, state_dict=sd, cond_stage=cond, unet_config=NARROW, vae_config=VAE_SMALL,
                                latent_size=16, resolution=128, **kw)
    image = torch.rand(2, 3, 128, 128, generator=torch.Generator().manual_seed(0))
    src, tgt = ['a photo of a cat', 'a tree'], ['a photo of a dog', 'a tree in winter']
    torch.manual_seed(123)
    z_ens = w.encode(image, src)
    img = w(z_ens, image, src, tgt).cpu()
    ora = dpm_encoder.LatentCycle(lambda x, t, c: unet_openai.unet_forward(usd, NARROW, x, t, c),
                                  lambda im: vae_kl.encode_moments(vsd, VAE_SMALL, im), lambda zz: vae_kl.decode(vsd, VAE_SMALL, zz), cond,
                                  channels=4, latent_size=16, resolution=128, **kw)
    torch.manual_seed(123)
    with torch.no_grad():
        z_ref = ora.encode(image, src)
        img_ref = ora.forward_all(z_ref, tgt)[0]
        img_x = ora.forward_all([z_ens[0].cpu()], tgt)[0]          # oracle decode of the engine's z
    rz = maxdiff(z_ens[0].cpu(), z_ref[0]) / float(z_ref[0].abs().max())
    print(f'sd wrapper: z {tuple(z_ens[0].shape)} rel|dz| {rz:.2e}  |d img| {maxdiff(img, img_ref):.2e}  cross |d img| {maxdiff(img, img_x):.2e}')
    assert len(z_ens) == 1 and z_ens[0].shape == z_ref[0].shape
    assert rz < 2e-4
    assert maxdiff(img, img_ref) < 1e-3
    assert maxdiff(img, img_x) < 1e-3
    with pytest.raises(AssertionError):
        w.encode(torch.rand(1, 3, 64, 64), ['x'])          # SDW:178 resolution check


def test_model_api_and_factory(eng):
    """TextUnsupervisedTranslation.forward keeps the reference signature and return tuple (text_unsupervised_translation.py:24-40)."""
    from cycle_diffusion_b200.models import TextUnsupervisedTranslation
    from cycle_diffusion_b200.wrappers import SyntheticTextEncoder
    usd = specs.synth_state_dict(specs.openai_unet_params(NARROW), 11)
    vsd = specs.synth_state_dict(specs.kl_vae_params(VAE_SMALL), 21)
    sd = {'model.diffusion_model.' + k: v for k, v in usd.items()}
    sd.update({'first_stage_model.' + k: v for k, v in vsd.items()})
    gan = dict(gan_type='SDStochasticText', source_model_type='synthetic', custom_steps=4, eta=0.1, white_box_steps=5, skip_steps=[1],
               encoder_unconditional_guidance_scales=[1], decoder_unconditional_guidance_scales=[2.0], n_trials=1)
    m = TextUnsupervisedTranslation(dict(gan=gan), engine=eng, state_dict=sd, cond_stage=SyntheticTextEncoder(48), unet_config=NARROW,
                                    vae_config=VAE_SMALL, latent_size=16, resolution=128).eval()
    image = torch.rand(1, 3, 128, 128)
    (orig, img), loss, losses = m(torch.tensor([0]), image, ['a'], ['b'])
    assert orig is image and img.shape == (1, 3, 128, 128) and loss.shape == (1,) and losses == {}
    assert torch.isfinite(img).all()


def test_ldm_wrapper_vs_oracle(eng):
    """LatentDiffStochasticTextWrapper (BASELINE config 4 class): posterior MEAN (latentdiff/.../ddpm.py:537-538), 2 ensemble
    members (two skip_steps) x 1 decoder scale, ranked by an injected scorer."""
    from cycle_diffusion_b200.wrappers import LatentDiffStochasticTextWrapper, SyntheticTextEncoder
    from oracle import dpm_encoder, unet_openai, vae_kl
    usd = specs.synth_state_dict(specs.openai_unet_params(NARROW), 11)
    vsd = specs.synth_state_dict(specs.kl_vae_params(VAE_SMALL), 21)
    sd = {'model.diffusion_model.' + k: v for k, v in usd.items()}
    sd.update({'first_stage_model.' + k: v for k, v in vsd.items()})
    cond = SyntheticTextEncoder(48)
    kw = dict(custom_steps=5, eta=0.1, white_box_steps=6, skip_steps=[1, 2], encoder_unconditional_guidance_scales=[1.0],
              decoder_unconditional_guidance_scales=[2.0], n_trials=1)
    ranker = lambda img, orig, et, dt: (None, -(img - orig).flatten(1).abs().mean(1))      # stand-in for DirectionalCLIP
    w = LatentDiffStochasticTextWrapper('synthetic', engine=eng, state_dict=sd, cond_stage=cond, unet_config=NARROW, vae_config=VAE_SMALL,
                                        latent_size=16, resolution=128, ranker=ranker, **kw)
    assert w.resolution == 128 and not w.generator.sample_posterior
    image = torch.rand(2, 3, 128, 128, generator=torch.Generator().manual_seed(3))
    torch.manual_seed(321)
    z_ens = w.encode(image, ['a', 'b'])
    img = w(z_ens, image.to(eng.device), ['a', 'b'], ['c', 'd']).cpu()
    ora = dpm_encoder.LatentCycle(lambda x, t, c: unet_openai.unet_forward(usd, NARROW, x, t, c),
                                  lambda im: vae_kl.encode_moments(vsd, VAE_SMALL, im), lambda zz: vae_kl.decode(vsd, VAE_SMALL, zz), cond,
                                  channels=4, latent_size=16, resolution=128, sample_posterior=False, **kw)
    torch.manual_seed(321)
    with torch.no_grad():
        z_ref = ora.encode(image, ['a', 'b'])
        imgs_ref = ora.forward_all(z_ref, ['c', 'd'])
    assert len(z_ens) == 2 and z_ens[0].shape[1] == 5 * 4 * 16 * 16 and z_ens[1].shape[1] == 4 * 4 * 16 * 16
    for a, b in zip(z_ens, z_ref):
        assert maxdiff(a.cpu(), b) / float(b.abs().max()) < 2e-4
    scores = torch.stack([ranker(i, image, None, None)[1] for i in imgs_ref], dim=1)
    best = scores.argmax(1)
    ref = torch.stack([imgs_ref[best[b].item()][b] for b in range(2)])
    print(f'ldm wrapper: |d img| {maxdiff(img, ref):.2e}')
    assert maxdiff(img, ref) < 1e-3


def test_pipeline_surface(eng):
    """CycleDiffusionPipeline.__call__ (Diffusers-style; unpinned surface): same-prompt cycle reproduces the input image's
    VAE reconstruction, strength maps to skip_steps, tuple / dataclass returns."""
    from cycle_diffusion_b200.pipeline import CycleDiffusionPipeline
    from cycle_diffusion_b200.wrappers import SDStochasticTextWrapper, SyntheticTextEncoder
    usd = specs.synth_state_dict(specs.openai_unet_params(NARROW), 11)
    vsd = specs.synth_state_dict(specs.kl_vae_params(VAE_SMALL), 21)
    sd = {'model.diffusion_model.' + k: v for k, v in usd.items()}
    sd.update({'first_stage_model.' + k: v for k, v in vsd.items()})
    w = SDStochasticTextWrapper('synthetic', custom_steps=4, eta=0.1, white_box_steps=5, skip_steps=[0], encoder_unconditional_guidance_scales=[1],
                                decoder_unconditional_guidance_scales=[1], n_trials=1, engine=eng, state_dict=sd, cond_stage=SyntheticTextEncoder(48),
                                unet_config=NARROW, vae_config=VAE_SMALL, latent_size=16, resolution=128)
    pipe = CycleDiffusionPipeline.from_wrapper(w)
    image = torch.rand(1, 3, 128, 128, generator=torch.Generator().manual_seed(4))
    gen = torch.Generator().manual_seed(9)
    out = pipe('a cat', 'a cat', image, strength=0.75, num_inference_steps=8, guidance_scale=1.0, source_guidance_scale=1.0, eta=0.1, generator=gen)
    # same prompt + same guidance: the cycle is the identity on the latent, so the output is decode(encode(image))
    g = w.generator
    gen = torch.Generator().manual_seed(9)
    mom = g.encode_first_stage(eng.shift_scale(image, -0.5, 2.0))
    x0 = eng.vae_posterior(mom, torch.randn(1, 4, 16, 16, generator=gen), 0.18215)
    rec = eng.shift_scale(g.decode_first_stage(x0), 1.0, 0.5).clamp(0, 1)
    assert out.images.shape == (1, 3, 128, 128)
    assert maxdiff(out.images.cpu(), rec.cpu()) < 1e-3
    tup = pipe(['a dog'], ['a cat'], image, num_inference_steps=4, return_dict=False, output_type='np')
    assert isinstance(tup, tuple) and tup[0].shape == (1, 128, 128, 3)
    with pytest.raises(ValueError):
        pipe('a', 'b', image, strength=1.5)


@pytest.mark.parametrize('tag', ['a', 'b'])
def test_lockstep_driver_vs_reference_fixture_and_two_phase(eng, tag):
    """cdx_cycle_lockstep (one U-Net call + one fused elementwise kernel per step, recovered noise consumed in registers):
    against the reference-generated fixture (DDIMSampler encode -> decode) and against the engine's own two-phase drivers."""
    from cycle_diffusion_b200.engine import UNet
    from cycle_diffusion_b200.schedule import DDIMSchedule
    g = golden('ddim_cycle_narrow')
    S, skip, wb, enc_scale, dec_scale, seed = [float(v) for v in g[f'cfg_{tag}']]
    S, skip, wb, seed = int(S), int(skip), int(wb), int(seed)
    sd = specs.synth_state_dict(specs.openai_unet_params(NARROW), 11)
    unet = UNet(eng, NARROW, 'openai').load_state_dict(sd)
    sched = DDIMSchedule(S, 0.1, skip)
    n_rec = min(sched.refine_steps, wb - skip - 1)
    if n_rec != sched.refine_steps:
        pytest.skip('lock-step needs every step recovered')
    torch.manual_seed(seed)
    noise = _encode_noise(sched, n_rec, g['x0'].shape)
    l0 = eng.launches
    out, z = unet.cycle_lockstep(g['x0'], g['c_src'], g['c_tgt'], g['uc'], enc_scale, dec_scale, sched, noise, return_z=True)
    torch.cuda.synchronize()
    l_lock = eng.launches - l0
    z2 = unet.latent_encode(g['x0'], g['c_src'], g['uc'], enc_scale, sched, n_rec, noise)
    out2 = unet.latent_decode(z2, g['c_tgt'], g['uc'], dec_scale, sched)
    zref = g[f'z_{tag}'].view(z.shape)
    rz = maxdiff(z.cpu(), zref) / float(zref.abs().max())
    d_ref = maxdiff(out.cpu(), g[f'tgt_{tag}'])
    d_two = maxdiff(out.cpu(), out2.cpu())
    rz_two = maxdiff(z.cpu(), z2.cpu()) / float(zref.abs().max())
    print(f'lockstep[{tag}]: rel|dz| vs reference {rz:.2e}  |d x| vs reference {d_ref:.2e}  vs two-phase: rel|dz| {rz_two:.2e} |d x| {d_two:.2e}'
          f'  bit-identical z {bool(torch.equal(z, z2))} x {bool(torch.equal(out, out2))}  launches {l_lock}')
    assert rz < 2e-4 and d_ref < 1e-3
    assert rz_two < 2e-5 and d_two < 1e-4


def test_pipeline_surface_vs_oracle(eng):
    """CycleDiffusionPipeline.__call__ (lock-step loop) against the ORACLE's restatement of the same computation
    (VAE encode -> posterior sample -> DPM-Encoder under the source prompt -> CFG decode under the target prompt -> VAE decode),
    same generator seed.  (The Diffusers class itself is not in /root/reference: the surface is unpinned, the arithmetic is not.)"""
    from cycle_diffusion_b200.pipeline import CycleDiffusionPipeline
    from cycle_diffusion_b200.wrappers import SDStochasticTextWrapper, SyntheticTextEncoder
    from oracle import dpm_encoder, unet_openai, vae_kl
    usd = specs.synth_state_dict(specs.openai_unet_params(NARROW), 11)
    vsd = specs.synth_state_dict(specs.kl_vae_params(VAE_SMALL), 21)
    sd = {'model.diffusion_model.' + k: v for k, v in usd.items()}
    sd.update({'first_stage_model.' + k: v for k, v in vsd.items()})
    cond = SyntheticTextEncoder(48)
    w = SDStochasticTextWrapper('synthetic', custom_steps=4, eta=0.1, white_box_steps=5, skip_steps=[0], encoder_unconditional_guidance_scales=[1],
                                decoder_unconditional_guidance_scales=[1], n_trials=1, engine=eng, state_dict=sd, cond_stage=cond,
                                unet_config=NARROW, vae_config=VAE_SMALL, latent_size=16, resolution=128)
    pipe = CycleDiffusionPipeline.from_wrapper(w)
    image = torch.rand(2, 3, 128, 128, generator=torch.Generator().manual_seed(4))
    S, strength, gs, sgs = 8, 0.75, 4.0, 1.0
    out = pipe(['a dog', 'a red car'], ['a cat', 'a blue car'], image, strength=strength, num_inference_steps=S, guidance_scale=gs,
               source_guidance_scale=sgs, eta=0.1, generator=torch.Generator().manual_seed(9)).images.cpu()
    out2 = pipe(['a dog', 'a red car'], ['a cat', 'a blue car'], image, strength=strength, num_inference_steps=S, guidance_scale=gs,
                source_guidance_scale=sgs, eta=0.1, generator=torch.Generator().manual_seed(9), two_phase=True).images.cpu()
    skip = S - int(S * strength)
    ora = dpm_encoder.LatentCycle(lambda x, t, c: unet_openai.unet_forward(usd, NARROW, x, t, c),
                                  lambda im: vae_kl.encode_moments(vsd, VAE_SMALL, im), lambda zz: vae_kl.decode(vsd, VAE_SMALL, zz), cond,
                                  custom_steps=S, eta=0.1, white_box_steps=S + 1, skip_steps=[skip], encoder_unconditional_guidance_scales=[sgs],
                                  decoder_unconditional_guidance_scales=[gs], n_trials=1, channels=4, latent_size=16, resolution=128)
    torch.manual_seed(9)
    with torch.no_grad():
        z_ref = ora.encode(image, ['a cat', 'a blue car'])
        ref = ora.forward_all(z_ref, ['a dog', 'a red car'])[0].clamp(0, 1)
    print(f'pipeline vs oracle: |d img| {maxdiff(out, ref):.2e}   lock-step vs two-phase {maxdiff(out, out2):.2e}')
    assert maxdiff(out, ref) < 1e-3
    assert maxdiff(out, out2) < 1e-4


def test_ensemble_batched_vs_oracle_member_by_member(eng):
    """SURVEY 8f-2: the ensemble of SDW:146-165 / 189-204 (n_trials x encoder scales x skips, then x decoder scales) with the members
    of one schedule batched along B (cdx_latent_loop_ens: per-sample guidance scales, conditioning and context K/V computed once).
    Every z and every image is compared with the CPU oracle's one-chain-at-a-time restatement, same seeds, same draw order; and with
    the wrapper's own sequential loops (ensemble_batch=None)."""
    from cycle_diffusion_b200.wrappers import SDStochasticTextWrapper, SyntheticTextEncoder
    from oracle import dpm_encoder, unet_openai, vae_kl
    usd = specs.synth_state_dict(specs.openai_unet_params(NARROW), 11)
    vsd = specs.synth_state_dict(specs.kl_vae_params(VAE_SMALL), 21)
    sd = {'model.diffusion_model.' + k: v for k, v in usd.items()}
    sd.update({'first_stage_model.' + k: v for k, v in vsd.items()})
    cond = SyntheticTextEncoder(48)
    kw = dict(custom_steps=6, eta=0.1, white_box_steps=7, skip_steps=[2, 3], encoder_unconditional_guidance_scales=[1.0, 3.0],
              decoder_unconditional_guidance_scales=[1.0, 3.0], n_trials=2)
    mk = lambda eb: SDStochasticTextWrapper('synthetic', engine=eng, state_dict=sd, cond_stage=cond, unet_config=NARROW, vae_config=VAE_SMALL,
                                            latent_size=16, resolution=128, ensemble_batch=eb, **kw)
    w, w_seq = mk(6), mk(None)
    image = torch.rand(2, 3, 128, 128, generator=torch.Generator().manual_seed(5))
    src, tgt = ['a photo of a cat', 'a tree'], ['a photo of a dog', 'a tree in winter']
    torch.manual_seed(77)
    z_ens = w.encode(image, src)
    imgs = [eng.shift_scale(i, 1.0, 0.5).cpu() for i in w.generate(z_ens, tgt)]
    torch.manual_seed(77)
    z_seq = w_seq.encode(image, src)
    imgs_seq = [eng.shift_scale(i, 1.0, 0.5).cpu() for i in w_seq.generate(z_seq, tgt)]
    ora = dpm_encoder.LatentCycle(lambda x, t, c: unet_openai.unet_forward(usd, NARROW, x, t, c),
                                  lambda im: vae_kl.encode_moments(vsd, VAE_SMALL, im), lambda zz: vae_kl.decode(vsd, VAE_SMALL, zz), cond,
                                  channels=4, latent_size=16, resolution=128, **kw)
    torch.manual_seed(77)
    with torch.no_grad():
        z_ref = ora.encode(image, src)
        imgs_ref = ora.forward_all(z_ref, tgt)
    assert len(z_ens) == len(z_ref) == 8 and len(imgs) == len(imgs_ref) == 16
    worst_z = worst_i = worst_s = 0.0
    for a, b, c_ in zip(z_ens, z_ref, z_seq):
        assert a.shape == b.shape
        worst_z = max(worst_z, maxdiff(a.cpu(), b) / float(b.abs().max()))
        worst_s = max(worst_s, maxdiff(a.cpu(), c_.cpu()) / float(b.abs().max()))
    for a, b, c_ in zip(imgs, imgs_ref, imgs_seq):
        worst_i = max(worst_i, maxdiff(a, b))
        worst_s = max(worst_s, maxdiff(a, c_))
    print(f'ensemble (8 encode x 2 decode members): rel|dz| {worst_z:.2e}  |d img| {worst_i:.2e}  batched vs sequential {worst_s:.2e}')
    assert worst_z < 2e-4 and worst_i < 1e-3 and worst_s < 1e-3
