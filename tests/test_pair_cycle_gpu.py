"""Two-model translation (UnsupervisedTranslation: two pixel DPMs or two unconditional LDMs) as one lock-step loop.

The lock-step drivers (cdx_pixel_cycle_lockstep, cdx_cycle_lockstep_pair) run each chain at batch B on its own network, exactly as
the two-phase encode -> z -> forward does, and consume the recovered noise in the same arithmetic, so their result must be
bit-identical to the two-phase one: these tests compare with torch.equal, not with a tolerance."""
import os
import re

import pytest
import torch

from cycle_diffusion_b200 import specs
from tests.common import golden, maxdiff

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW_SYMBOLS = ('cdx_pixel_cycle_lockstep', 'cdx_cycle_lockstep_pair')

gpu = pytest.mark.gpu

PIXEL_CASES = {'ddim': dict(sample_type='ddim', eta=0.1, custom_steps=10, es_steps=10),
               'ddpm': dict(sample_type='ddpm', eta=None, custom_steps=20, es_steps=6),
               'ddim_refine': dict(sample_type='ddim', eta=0.1, custom_steps=10, es_steps=10, refine_steps=3, refine_iterations=2)}
DDPM_SMALL = dict(image_size=32, in_channels=3, out_channels=3, model_channels=32, num_res_blocks=2, channel_mult=(1, 2, 2), attention_resolutions=(2,))
UNCOND_SMALL = dict(in_channels=3, out_channels=3, model_channels=32, attention_resolutions=(2, 4), num_res_blocks=1,
                    channel_mult=(1, 2, 2), num_head_channels=16, context_dim=0)
VQ_SMALL = dict(ch=32, ch_mult=(1, 2, 4), num_res_blocks=1, in_channels=3, out_ch=3, z_channels=3, embed_dim=3, vq=True, n_embed=256)


def test_new_entry_points_exported_and_declared():
    """CPU: both drivers are declared in cdx.h, exported by libcdx.so and bound with a ctypes signature."""
    from cycle_diffusion_b200 import _cabi
    txt = re.sub(r'/\*.*?\*/', '', open(os.path.join(ROOT, 'include', 'cdx.h')).read(), flags=re.S)
    for s in NEW_SYMBOLS:
        assert re.search(r'\b' + s + r'\s*\(', txt), f'{s} not declared in cdx.h'
        assert hasattr(_cabi.lib, s), f'{s} not exported by libcdx.so'
        assert s in _cabi.SIGNATURES
    assert _cabi.lib.cdx_abi_version() == 2


# ------------------------------------------------------------------------------------------------ fixtures
@pytest.fixture(scope='module')
def engines():
    from cycle_diffusion_b200.engine import Engine
    return Engine(0), Engine(0)


@pytest.fixture(scope='module')
def iddpm(engines):
    """i-DDPM 64x64 U-Nets: source (seed 31) on engine 0, target (seed 32) on engine 0 and, separately, on engine 1."""
    from cycle_diffusion_b200.engine import UNet
    eng, eng2 = engines
    cfg = specs.iddpm_config(64)
    sd31 = specs.synth_state_dict(specs.iddpm_unet_params(cfg), 31)
    sd32 = specs.synth_state_dict(specs.iddpm_unet_params(cfg), 32)
    return dict(src=UNet(eng, cfg, 'iddpm').load_state_dict(sd31),
                tgt={'shared': UNet(eng, cfg, 'iddpm').load_state_dict(sd32), 'separate': UNet(eng2, cfg, 'iddpm').load_state_dict(sd32)})


def _pixel_model(kw, src_net, tgt_net, rng='cpu', R=64, src_kw=None, tgt_kw=None):
    from cycle_diffusion_b200.models import UnsupervisedTranslation
    gan = dict(gan_type='DDPM_DDIM', source_model_type=f'afhqcat{R}', target_model_type=f'afhqdog{R}', **kw)
    return UnsupervisedTranslation(dict(gan=gan), source_kwargs=dict(unet=src_net, image_size=R, rng=rng, **(src_kw or {})),
                                   target_kwargs=dict(unet=tgt_net, image_size=R, rng=rng, **(tgt_kw or {}))).eval()


def _forward(m, image, seed):
    torch.manual_seed(seed)
    (_, img), _, _ = m(torch.tensor([0]), original_image=image)
    return img


def _two_phase(m, image, seed):
    torch.manual_seed(seed)
    z = m.source_gan_wrapper.encode(image=image)
    return m.target_gan_wrapper(z=z)


def _image(B, R, seed):
    return torch.rand(B, 3, R, R, generator=torch.Generator().manual_seed(seed))


# ------------------------------------------------------------------------------------------------ pixel DPMs
@gpu
@pytest.mark.parametrize('engines_mode', ['shared', 'separate'])
@pytest.mark.parametrize('B', [1, 3])
@pytest.mark.parametrize('rng', ['cpu', 'cuda'])
@pytest.mark.parametrize('case', list(PIXEL_CASES))
def test_pixel_pair_equals_two_phase(iddpm, case, rng, B, engines_mode):
    m = _pixel_model(PIXEL_CASES[case], iddpm['src'], iddpm['tgt'][engines_mode], rng)
    assert m.source_gan_wrapper.pair_cycle_applies(m.target_gan_wrapper)
    image = _image(B, 64, 7 + B)
    out = _forward(m, image, 1234)
    ref = _two_phase(m, image, 1234)
    assert out.shape == ref.shape == (B, 3, 64, 64)
    assert torch.equal(out, ref), f'lock-step vs two-phase max |d| {maxdiff(out.cpu(), ref.cpu()):.3e}'


@gpu
def test_pixel_pair_on_the_ddpm_family_equals_two_phase(engines):
    """Ho-et-al DDPM U-Nets (CDX_UNET_DDPM, 3 output channels: no learn_sigma split), one per engine."""
    from cycle_diffusion_b200.engine import UNet
    eng, eng2 = engines
    src = UNet(eng, DDPM_SMALL, 'ddpm').load_state_dict(specs.synth_state_dict(specs.ddpm_unet_params(DDPM_SMALL), 61))
    tgt = UNet(eng2, DDPM_SMALL, 'ddpm').load_state_dict(specs.synth_state_dict(specs.ddpm_unet_params(DDPM_SMALL), 62))
    m = _pixel_model(PIXEL_CASES['ddim'], src, tgt, R=32)
    assert m.source_gan_wrapper.pair_cycle_applies(m.target_gan_wrapper)
    image = _image(2, 32, 2)
    out, ref = _forward(m, image, 11), _two_phase(m, image, 11)
    assert torch.equal(out, ref), f'max |d| {maxdiff(out.cpu(), ref.cpu()):.3e}'


@gpu
@pytest.mark.parametrize('tag', list(PIXEL_CASES))
def test_pixel_pair_vs_reference_fixture(iddpm, tag):
    """Both sides with the fixture's weights (seed 31): the lock-step cycle reproduces the unmodified reference wrapper's
    encode -> forward (tolerances of test_cycle_gpu.test_pixel_wrapper_vs_reference_fixture)."""
    g = golden('pixel_cycle_iddpm64')
    m = _pixel_model(PIXEL_CASES[tag], iddpm['src'], iddpm['src'])
    assert m.source_gan_wrapper.pair_cycle_applies(m.target_gan_wrapper)
    img = _forward(m, g['image'], 2000).cpu()
    tol = max(1e-3, 8 * float(g[f'sens_{tag}']))
    print(f'pixel pair[{tag}]: |d img| vs reference {maxdiff(img, g[f"img_{tag}"]):.2e} (tol {tol:.1e})')
    assert maxdiff(img, g[f'img_{tag}']) < tol


@gpu
@pytest.mark.parametrize('case', ['ddim', 'ddpm'])
def test_pixel_pair_z_out_equals_pixel_encode(iddpm, case):
    from cycle_diffusion_b200.schedule import PixelSchedule
    kw = PIXEL_CASES[case]
    sched = PixelSchedule(kw['sample_type'], kw['custom_steps'], kw['es_steps'], kw['eta'], 999)
    src, tgt = iddpm['src'], iddpm['tgt']['separate']
    g = torch.Generator().manual_seed(5)
    x = torch.rand(3, 3, 64, 64, generator=g) * 2 - 1
    noise = torch.randn((kw['es_steps'], 3, 3, 64, 64), generator=g)
    last = torch.randn((1, 3, 3, 64, 64), generator=g)
    out, z = src.pixel_cycle_lockstep(tgt, x, sched, noise, last, return_z=True)
    z2 = src.pixel_encode(x, sched, noise)
    out2 = tgt.pixel_decode(z2, sched, last_noise=last)
    assert torch.equal(z, z2), f'z max |d| {maxdiff(z.cpu(), z2.cpu()):.3e}'
    assert torch.equal(out, out2)
    assert torch.equal(src.pixel_cycle_lockstep(tgt, x, sched, noise, last), out)     # without z_out: same result


# ------------------------------------------------------------------------------------------------ unconditional LDMs
def _ldm_sd(seed):
    sd = {'model.diffusion_model.' + k: v for k, v in specs.synth_state_dict(specs.openai_unet_params(UNCOND_SMALL), seed).items()}
    sd.update({'first_stage_model.' + k: v for k, v in specs.synth_state_dict(specs.kl_vae_params(VQ_SMALL), seed + 1).items()})
    return sd


def _ldm_model(eng_src, eng_tgt, S=6, wb=7, refine=2, tgt_kw=None):
    from cycle_diffusion_b200.models import UnsupervisedTranslation
    from cycle_diffusion_b200.schedule import ldm_alphas_cumprod
    gan = dict(gan_type='LatentDiffStochastic', source_model_type='ffhq256', target_model_type='celeba256', custom_steps=S, eta=0.1,
               white_box_steps=wb, refine_steps=refine)
    common = dict(unet_config=UNCOND_SMALL, vae_config=VQ_SMALL, latent_size=16, resolution=64, alphas_cumprod=ldm_alphas_cumprod())
    return UnsupervisedTranslation(dict(gan=gan), source_kwargs=dict(engine=eng_src, state_dict=_ldm_sd(41), **common),
                                   target_kwargs=dict(engine=eng_tgt, state_dict=_ldm_sd(51), **common, **(tgt_kw or {}))).eval()


@gpu
@pytest.mark.parametrize('engines_mode', ['shared', 'separate'])
def test_ldm_pair_equals_two_phase(engines, engines_mode):
    eng, eng2 = engines
    m = _ldm_model(eng, eng if engines_mode == 'shared' else eng2)
    src, tgt = m.source_gan_wrapper, m.target_gan_wrapper
    assert src.pair_cycle_applies(tgt)
    image = _image(2, 64, 3)
    out, ref = _forward(m, image, 77), _two_phase(m, image, 77)
    assert out.shape == (2, 3, 64, 64)
    assert torch.equal(out, ref), f'max |d| {maxdiff(out.cpu(), ref.cpu()):.3e}'
    # the driver's optional z equals the DPM-Encoder's
    sched = src._sched()
    x0 = torch.randn(2, 3, 16, 16, generator=torch.Generator().manual_seed(1))
    noise = torch.randn((sched.refine_steps + 1, 2, 3, 16, 16), generator=torch.Generator().manual_seed(2))
    y, z = src.generator.unet.cycle_lockstep_pair(tgt.generator.unet, x0, None, None, None, 1.0, 1.0, sched, noise, return_z=True)
    z2 = src.generator.unet.latent_encode(x0, None, None, 1.0, sched, sched.refine_steps, noise)
    assert torch.equal(z, z2)
    assert torch.equal(y, tgt.generator.unet.latent_decode(z2, None, None, 1.0, sched))


# ------------------------------------------------------------------------------------------------ fallback to two-phase
@gpu
def test_ldm_fallback_when_not_every_step_is_recovered(engines):
    eng, eng2 = engines
    m = _ldm_model(eng, eng2, S=6, wb=4)            # white_box_steps - 1 < 6 steps: the decode draws fresh noise for 3 steps
    assert not m.source_gan_wrapper.pair_cycle_applies(m.target_gan_wrapper)
    image = _image(1, 64, 4)
    assert torch.equal(_forward(m, image, 5), _two_phase(m, image, 5))


@gpu
def test_pixel_fallback_on_mismatched_schedules(iddpm):
    src, tgt = iddpm['src'], iddpm['tgt']['separate']
    kw = PIXEL_CASES['ddim']
    m = _pixel_model(kw, src, tgt, tgt_kw=dict(custom_steps=12))           # same es_steps, different step pairs
    assert not m.source_gan_wrapper.pair_cycle_applies(m.target_gan_wrapper)
    image = _image(2, 64, 6)
    assert torch.equal(_forward(m, image, 9), _two_phase(m, image, 9))
    m = _pixel_model(kw, src, tgt, tgt_kw=dict(es_steps=8))                # z of 10 steps does not fit a target of 8: both paths refuse
    assert not m.source_gan_wrapper.pair_cycle_applies(m.target_gan_wrapper)
    with pytest.raises(RuntimeError):
        _forward(m, image, 9)
    with pytest.raises(RuntimeError):
        _two_phase(m, image, 9)


# ------------------------------------------------------------------------------------------------ work and memory
@gpu
@pytest.mark.parametrize('engines_mode', ['shared', 'separate'])
def test_pixel_pair_one_kernel_per_step_besides_the_unets(engines, iddpm, engines_mode):
    from cycle_diffusion_b200.schedule import PixelSchedule
    src, tgt = iddpm['src'], iddpm['tgt'][engines_mode]
    engs = list({id(e): e for e in (src.engine, tgt.engine)}.values())
    count = lambda: sum(e.launches for e in engs)
    B, n = 2, 10
    sched = PixelSchedule('ddim', n, n, 0.1, 999)
    x = torch.rand(B, 3, 64, 64) * 2 - 1
    t = torch.full((B,), 999.0)
    unet_launches = []
    for net in (src, tgt):
        net(x, t)
        torch.cuda.synchronize()
        l0 = count()
        net(x, t)
        torch.cuda.synchronize()
        unet_launches.append(count() - l0)
    u_src, u_tgt = unet_launches
    noise = torch.randn(n, B, 3, 64, 64)
    l0 = count()
    src.pixel_cycle_lockstep(tgt, x, sched, noise, None)
    torch.cuda.synchronize()
    lock = count() - l0
    l0 = count()
    tgt.pixel_decode(src.pixel_encode(x, sched, noise), sched)
    torch.cuda.synchronize()
    two = count() - l0
    other_lock = lock - (n - 1) * (u_src + u_tgt) - u_tgt
    other_two = two - (n - 1) * u_src - n * u_tgt
    print(f'launches per cycle besides the U-Nets ({u_src} + {u_tgt} per forward): lock-step {other_lock}, two-phase {other_two}')
    # q_sample, one fused kernel per lock-step iteration, the final target-only step
    assert other_lock == 1 + (n - 1) + 1
    assert other_two == 1 + 2 * (n - 1) + n


@gpu
def test_pixel_pair_peak_memory_saves_z(iddpm):
    B, n = 2, 50
    m = _pixel_model(dict(sample_type='ddim', eta=0.1, custom_steps=n, es_steps=n), iddpm['src'], iddpm['tgt']['separate'], 'cuda')
    image = _image(B, 64, 8)
    z_bytes = B * n * 3 * 64 * 64 * 4
    _forward(m, image, 1)          # warm both paths (workspace growth is outside torch's allocator, but keep the runs alike)
    _two_phase(m, image, 1)
    peaks = {}
    for name, fn in (('lock', _forward), ('two', _two_phase)):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        out = fn(m, image, 1)
        torch.cuda.synchronize()
        peaks[name] = torch.cuda.max_memory_allocated() - base
        del out
    print(f'peak torch memory: lock-step {peaks["lock"] / 2**20:.2f} MiB, two-phase {peaks["two"] / 2**20:.2f} MiB, z {z_bytes / 2**20:.2f} MiB')
    assert peaks['two'] - peaks['lock'] >= 0.9 * z_bytes
