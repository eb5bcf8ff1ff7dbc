#!/usr/bin/env python
"""bench.py -- images/sec of the CycleDiffusion hot path on N B200s of one node.

One "step" = one full cycle over one batch of synthetic (image, source-text, target-text) triplets per GPU.  Default workload
= BASELINE.json configs[1] (the configuration the metric is quoted on):
    VAE encode (+posterior sample) -> 50-step DPM-Encoder under the source condition (scale 1)
    -> 50-step decode under the target condition with classifier-free guidance 7.5 -> VAE decode -> (x+1)/2
on the Stable Diffusion v1-4 topology (859.5 M-param U-Net, KL-f8 VAE, random-init weights -- there are no checkpoints
offline), 512x512, batch 4 per GPU (README.md:153), fp32 end to end.  `--config 4` = LDM text2img-large 256x256, 50 steps,
batch 16; `--config 5` = cat->dog with two improved-DDPM 256x256 U-Nets, 250-step encode / decode, batch 8 per GPU.

    python bench.py --gpus 1 --steps K --warmup W [--config 2|4|5]      # our engine
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...                                # the reference's CPU path (oracle port), rank 0 only
    python bench.py ... --dump-outputs DIR                              # also save the last timed step's images as DIR/images.npy

Prints ONE JSON line.  `value` is timed with inputs resident in HBM; `e2e` goes through the drop-in wrapper API with HOST
buffers (H2D of image / conditioning / noise and D2H of the result inside the timed region).  `roofline` comes from a separate
untimed profiling pass (CUDA events around every launch of each kernel family, inside libcdx); `cpu_baseline` times the CPU
oracle on a bounded sample on rank 0; `fast_path` is the separately reported reduced-precision mode (mma_mode 4) with its
measured |delta pixel| against the fp32-faithful result of the same short cycle.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

if os.environ.get('NCCL_DEBUG', '').upper() == 'VERSION':     # NCCL prints its banner to stdout: keep stdout = the one JSON line
    os.environ['NCCL_DEBUG'] = 'WARN'
import numpy as np  # noqa: E402
import torch  # noqa: E402

UNIT = 'images/s'
ETA = 0.1

# per-configuration constants (BASELINE.md section 2: FLOPs per image and per U-Net sample-forward)
CONFIGS = {
    2: dict(name='BASELINE configs[1]: Stable Diffusion v1-4 512x512, 50-step DPMEncoder (scale 1) + 50-step CFG decode (scale 7.5), batch 4 per GPU',
            metric='images/sec (512x512, 50-step encode+decode)', kind='latent', ctx=768, res=512, lat=64, B=4, steps=50, enc_scale=1.0,
            dec_scale=7.5, sample_posterior=True, tflop_per_image=124.1, unet_gflop=803.27),
    4: dict(name='BASELINE configs[3]: LDM text2img-large 256x256, 50-step DPMEncoder (scale 1) + 50-step CFG decode (scale 7.5), batch 16 per GPU',
            metric='images/sec (256x256 LDM text2img-large, 50-step encode+decode)', kind='latent', ctx=1280, res=256, lat=32, B=16, steps=50,
            enc_scale=1.0, dec_scale=7.5, sample_posterior=False, tflop_per_image=28.2, unet_gflop=182.07),
    5: dict(name='BASELINE configs[4]: unpaired cat->dog, two improved-DDPM 256x256 U-Nets (random-init), 250-step DDIM(eta 0.1) encode / decode, '
                 'batch 8 per GPU', metric='images/sec (256x256 pixel DDPM cat->dog, 250-step encode+decode)', kind='pixel', res=256, B=8, steps=250,
            tflop_per_image=193.6, unet_gflop=387.93),
}


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=p['hbm_gbs'], tflops=p['bf16_tflops'], tflops_sustained=p.get('bf16_tflops_sustained', p['bf16_tflops']),
                    source='measured (MEASURED_PEAKS.json: copy GB/s, cuBLAS bf16 TF/s)')
    return dict(hbm_gbs=6650.0, tflops=1590.0, tflops_sustained=1400.0, source='fallback (B200_PROFILING.md)')


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
            'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={q}', '--format=csv,noheader,nounits', '-lms', '200'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace('.', '').isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith('active')})
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': reasons, 'samples': len(sm)}


def synthetic_inputs(cfg, B, seed=0):
    """SURVEY.md 8d: image U[0,1] (seed 0), conditioning N(0,1) [B,77,D] (seed 1)."""
    g0, g1 = torch.Generator().manual_seed(seed), torch.Generator().manual_seed(1 + seed)
    image = torch.rand(B, 3, cfg['res'], cfg['res'], generator=g0)
    if cfg['kind'] != 'latent':
        return image, None, None, None
    D = cfg['ctx']
    c_src = torch.randn(B, 77, D, generator=g1)
    c_tgt = torch.randn(B, 77, D, generator=g1)
    uc = torch.randn(1, 77, D, generator=g1).expand(B, 77, D).contiguous()
    return image, c_src, c_tgt, uc


def encode_noise(sched, n_rec, shape, gen):
    noise = torch.zeros((n_rec + 1,) + tuple(shape))
    noise[0] = torch.randn(shape, generator=gen)
    for i in range(n_rec):
        if sched.refine_steps - 1 - i != 0:
            noise[1 + i] = torch.randn(shape, generator=gen)
    return noise


def timed(eng, fn, steps, warmup, world, dist):
    """-> (ms of the `steps` timed calls, launches they issued, what the last timed call returned)."""
    d = eng.device
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    l0 = eng.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=d)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item()), eng.launches - l0, out


def dump_outputs(path, **arrays):
    """Each array -> path/<name>.npy (float32), so that two builds can be compared output for output."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + '.npy'), a.detach().float().cpu().numpy())


def time_call(fn, reps=3, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def family_report(eng, fn, pk):
    """Per-kernel-family CUDA-event timing of one call of `fn` (untimed pass)."""
    eng.profile(True)
    fn()
    families = eng.profile_read()
    eng.profile(False)
    for v in families.values():
        if v['flops'] == 0 and v['bytes'] > 0 and v['ms'] > 0:
            v['gbs'] = round(v['bytes'] / (v['ms'] * 1e-3) / 1e9, 1)
            v['frac_hbm'] = round(v['gbs'] / pk['hbm_gbs'], 4)
        if v['flops'] and v['ms'] > 0:
            v['tflops'] = round(v['flops'] / (v['ms'] * 1e-3) / 1e12, 2)
        v['ms'] = round(v['ms'], 3)
    return families


def roofline_of(families, pk, value, tflop_per_image, mma_label):
    tensor_fams = {k: v for k, v in families.items() if v['flops'] > 0}
    if not tensor_fams:
        return None
    top = max(tensor_fams, key=lambda k: tensor_fams[k]['ms'])
    f = tensor_fams[top]
    ach = f['flops'] / (f['ms'] * 1e-3) / 1e12
    traffic = None      # DRAM bytes of one captured launch of this family (ncu --set full; profiles/ncu_traffic.json)
    try:
        with open(os.path.join(ROOT, 'profiles', 'ncu_traffic.json')) as fh:
            traffic = json.load(fh).get(top)
    except (OSError, ValueError):
        pass
    return {'kernel': top, 'bound': 'tensor', 'achieved': round(ach, 2), 'peak': pk['tflops_sustained'], 'unit': 'TFLOP/s',
            'frac': round(ach / pk['tflops_sustained'], 4),
            # the fp32-faithful path issues 3 fp16 MMAs per product (hi*hi + lo*hi + hi*lo): its own ceiling is peak / 3
            'frac_of_split_ceiling': round(ach / (pk['tflops_sustained'] / 3.0), 4), 'traffic': traffic, 'launches_per_call': f['launches'],
            'avg_launch_ms': round(f['ms'] / f['launches'], 4),
            'peak_source': pk['source'] + f' -- sustained bf16 dense; this path is {mma_label} (see DESIGN.md)',
            'whole_job_tflops': round(value * tflop_per_image, 2)}


MMA_LABELS = {None: 'tcgen05 3x fp16-split (fp32-faithful)', 0: 'ffma-fp32', 1: 'tcgen05 3x fp16-split (fp32-faithful)', 2: 'tcgen05 3x fp16-split, unfused attention',
              3: 'tcgen05 3xTF32 (fp32-faithful, round-1 scheme)', 4: 'tcgen05 1x fp16 (FAST PATH, not fp32-faithful)'}


# ================================================================================================ our arm
def run_ours(args):
    import torch.distributed as dist
    from cycle_diffusion_b200 import specs
    from cycle_diffusion_b200.engine import Engine, UNet, VAE
    from cycle_diffusion_b200.schedule import DDIMSchedule, PixelSchedule
    from cycle_diffusion_b200.wrappers import DDPMDDIMWrapper, LatentDiffStochasticTextWrapper, SDStochasticTextWrapper, _LatentGenerator

    cfg = CONFIGS[args.config]
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    assert world == args.gpus, f'--gpus {args.gpus} but WORLD_SIZE={world}'
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    eng = Engine(local)
    if args.mma is not None:
        eng.set_mma_mode(args.mma)
    latent = cfg['kind'] == 'latent'
    B, RES, S = cfg['B'], cfg['res'], cfg['steps']
    # frozen weights: rank 0 builds them, one NCCL broadcast of the packed blobs over NVLink, no other collective
    t0 = time.time()
    if latent:
        ucfg, vcfg = specs.sd_unet_config(cfg['ctx']), specs.kl_f8_config()
        nets = [UNet(eng, ucfg, 'openai'), VAE(eng, vcfg)]
        if rank == 0:
            nets[0].load_state_dict(specs.synth_state_dict(specs.openai_unet_params(ucfg), 1234))
            nets[1].load_state_dict(specs.synth_state_dict(specs.kl_vae_params(vcfg), 1235))
    else:
        icfg = specs.iddpm_config(RES)
        nets = [UNet(eng, icfg, 'iddpm'), UNet(eng, icfg, 'iddpm')]      # source (cat) and target (dog) models
        if rank == 0:
            nets[0].load_state_dict(specs.synth_state_dict(specs.iddpm_unet_params(icfg), 1234))
            nets[1].load_state_dict(specs.synth_state_dict(specs.iddpm_unet_params(icfg), 4321))
    bcast_ms = None
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for net in nets:
            dist.broadcast(net.blob_tensor(), src=0)
        e1.record()
        torch.cuda.synchronize()
        bcast_ms = e0.elapsed_time(e1)
        if rank != 0:
            for net in nets:
                net.adopt_blob()
    load_s = time.time() - t0

    image, c_src, c_tgt, uc = synthetic_inputs(cfg, B, seed=rank)
    d = eng.device
    gen = torch.Generator().manual_seed(7 + rank)
    pk = peaks()
    extra, stage_ms, unet_ms = {}, None, {}

    if latent:
        unet, vae = nets
        LAT = cfg['lat']
        sched = DDIMSchedule(S, ETA, 0)
        n_rec = sched.refine_steps
        post_noise = torch.randn(B, 4, LAT, LAT, generator=gen) if cfg['sample_posterior'] else None
        enc_noise = encode_noise(sched, n_rec, (B, 4, LAT, LAT), gen)
        dev = dict(image=image.to(d), c_src=c_src.to(d), c_tgt=c_tgt.to(d), uc=uc.to(d), noise=enc_noise.to(d),
                   post=post_noise.to(d) if post_noise is not None else None)

        def cycle_resident(lockstep=True, steps_sched=sched, noise=None):
            x = eng.shift_scale(dev['image'], -0.5, 2.0)
            x0 = eng.vae_posterior(vae.encode_moments(x), dev['post'], 0.18215)
            nz = dev['noise'] if noise is None else noise
            if lockstep:
                s = unet.cycle_lockstep(x0, dev['c_src'], dev['c_tgt'], dev['uc'], cfg['enc_scale'], cfg['dec_scale'], steps_sched, nz)
            else:
                z = unet.latent_encode(x0, dev['c_src'], dev['uc'], cfg['enc_scale'], steps_sched, steps_sched.refine_steps, nz)
                s = unet.latent_decode(z, dev['c_tgt'], dev['uc'], cfg['dec_scale'], steps_sched)
            return eng.shift_scale(vae.decode(eng.affine(s, 1. / 0.18215, 0.0)), 1.0, 0.5)

        # the drop-in wrapper over the SAME engine objects, fed with host tensors
        class _Cond:
            def __call__(self, texts):
                return pinned['uc'] if texts[0] == '' else (pinned['c_src'] if texts[0] == 'src' else pinned['c_tgt'])
        genr = _LatentGenerator(eng, unet, vae, _Cond(), 4, LAT, 0.18215, cfg['sample_posterior'])
        wcls = SDStochasticTextWrapper if args.config == 2 else LatentDiffStochasticTextWrapper
        wrap = wcls('synthetic', custom_steps=S, eta=ETA, white_box_steps=S + 1, skip_steps=[0],
                    encoder_unconditional_guidance_scales=[cfg['enc_scale']], decoder_unconditional_guidance_scales=[cfg['dec_scale']],
                    n_trials=1, generator=genr, resolution=RES)
        # the reference's model API over the same wrapper (text_unsupervised_translation.py:24-40): what Trainer.prediction_step calls
        from cycle_diffusion_b200.models import TextUnsupervisedTranslation
        model = TextUnsupervisedTranslation.__new__(TextUnsupervisedTranslation)
        torch.nn.Module.__init__(model)
        model.gan_wrapper = wrap
        model.eval()
        sample_id = torch.arange(B)
        pinned = {k: v.pin_memory() for k, v in dict(image=image, c_src=c_src, c_tgt=c_tgt, uc=uc).items()}
        out_host = torch.empty(B, 3, RES, RES).pin_memory()
        h2d = [4 * (image.numel() + 4 * c_src.numel() + (post_noise.numel() if post_noise is not None else 0) + enc_noise.numel())]
        api = (f'TextUnsupervisedTranslation.forward(sample_id, image, encode_text, decode_text) over {wcls.__name__} '
               '(single-member ensemble -> wrapper.cycle: lock-step loop); host tensors in, pinned host tensor out')

        def cycle_e2e(two_phase=False):
            torch.manual_seed(99)
            img_d = pinned['image'].to(d, non_blocking=True)
            if two_phase:           # the wrapper's own two calls (SDW:169-249): encode -> z -> forward
                z = wrap.encode(img_d, B * ['src'])
                img = wrap(z, img_d, B * ['src'], B * ['tgt'])
            else:
                (_, img), _, _ = model(sample_id, img_d, B * ['src'], B * ['tgt'])
            out_host.copy_(img, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            return img
    else:
        src, tgt = nets
        psched = PixelSchedule('ddim', S, S, ETA, 999)
        n_rec = S - 1
        # the first draw from the device's default generator, which starts from torch's fixed default seed: the same in every run
        noise_dev = torch.randn(n_rec + 1, B, 3, RES, RES, device=d)       # resident arm: noise lives in HBM (1.5 GB at B=8)
        last_dev = torch.zeros(1, B, 3, RES, RES, device=d)
        img_dev = image.to(d)

        def cycle_resident():
            x = eng.shift_scale(img_dev, -0.5, 2.0)
            z = src.pixel_encode(x, psched, noise_dev)
            return eng.shift_scale(tgt.pixel_decode(z, psched, last_noise=last_dev), 1.0, 0.5)

        kw = dict(sample_type='ddim', custom_steps=S, es_steps=S, eta=ETA)
        w_src = DDPMDDIMWrapper('cat256', unet=src, image_size=RES, rng='cuda', **kw)
        w_tgt = DDPMDDIMWrapper('dog256', unet=tgt, image_size=RES, rng='cuda', **kw)
        pinned = {'image': image.pin_memory()}
        out_host = torch.empty(B, 3, RES, RES).pin_memory()
        h2d = [4 * image.numel()]
        api = 'DDPMDDIMWrapper(source).encode -> DDPMDDIMWrapper(target).forward (unsupervised_translation.py:48-49), host image in / out, ' \
              "rng='cuda' (the reference-reproducible CPU draws would add 1.5 GB of host randn + H2D per batch)"

        def cycle_e2e():
            img_d = pinned['image'].to(d, non_blocking=True)
            z = w_src.encode(img_d)
            img = w_tgt(z)
            out_host.copy_(img, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            return img

    clocks = ClockSampler(local)
    clocks.start()
    ms_total, launches, images = timed(eng, cycle_resident, args.steps, args.warmup, world, dist)
    clk = clocks.stop()
    # rank 0's inputs are those of the single-GPU run, so its images are comparable across --gpus
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, images=images)
    e2e_steps = max(1, min(args.steps, 2))
    ms_e2e, _, _ = timed(eng, cycle_e2e, e2e_steps, 1, world, dist)
    value = world * B * args.steps / (ms_total / 1e3)
    e2e_value = world * B * e2e_steps / (ms_e2e / 1e3)

    # ---- untimed extra passes on rank 0: ms per U-Net call at the batches actually launched, per-family roofline, stage breakdown,
    # lock-step driver, fast path
    roof, families, norm_probe = None, {}, None
    if rank == 0:
        if latent:
            LAT = cfg['lat']
            t1 = torch.full((B,), 501., device=d)
            x1 = torch.randn(B, 4, LAT, LAT, device=d)
            x2, t2, ctx2 = torch.cat([x1, x1]), torch.cat([t1, t1]), torch.cat([dev['uc'], dev['c_tgt']])
            unet_ms[f'batch{B}'] = round(time_call(lambda: unet(x1, t1, dev['c_src'])), 2)
            unet_ms[f'cfg_batch{2 * B}'] = round(time_call(lambda: unet(x2, t2, ctx2)), 2)
            x3, t3, ctx3 = torch.cat([x1, x1, x1]), torch.cat([t1, t1, t1]), torch.cat([dev['c_src'], dev['uc'], dev['c_tgt']])
            unet_ms[f'lockstep_batch{3 * B}'] = round(time_call(lambda: unet(x3, t3, ctx3)), 2)
            families = family_report(eng, lambda: unet(x2, t2, ctx2), pk)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
            ev[0].record()
            x_ = eng.shift_scale(dev['image'], -0.5, 2.0)
            x0_ = eng.vae_posterior(vae.encode_moments(x_), dev['post'], 0.18215)
            ev[1].record()
            z_ = unet.latent_encode(x0_, dev['c_src'], dev['uc'], cfg['enc_scale'], sched, n_rec, dev['noise'])
            ev[2].record()
            s_ = unet.latent_decode(z_, dev['c_tgt'], dev['uc'], cfg['dec_scale'], sched)
            ev[3].record()
            ref_img = eng.shift_scale(vae.decode(eng.affine(s_, 1. / 0.18215, 0.0)), 1.0, 0.5)
            ev[4].record()
            torch.cuda.synchronize()
            stage_ms = {k: round(ev[i].elapsed_time(ev[i + 1]), 1) for i, k in
                        enumerate(['vae_encode', f'dpm_encode_{S}x_unet_b{B}', f'decode_{S}x_unet_b{2 * B}', 'vae_decode'])}
            # the headline runs the lock-step driver (one 3B-batch U-Net call per step, no z buffer); the reference-shaped two-phase
            # path (encode -> z -> decode, stage_ms above) is timed beside it, with the agreement of the two results
            ms_two = time_call(lambda: cycle_resident(lockstep=False), reps=1, warm=1)
            lock_img = cycle_resident(lockstep=True)
            ms_e2e_two = time_call(lambda: cycle_e2e(two_phase=True), reps=1, warm=1)
            extra['two_phase'] = {'images_per_s': round(B / (ms_two / 1e3), 4), 'ms_per_step': round(ms_two, 1),
                                  'e2e_images_per_s_wrapper_encode_forward': round(B / (ms_e2e_two / 1e3), 4),
                                  'max_abs_diff_lockstep_vs_two_phase': float((lock_img - ref_img).abs().max())}
            # fast path (mma_mode 4: hi*hi term only): same full cycle, |delta pixel| against the fp32-faithful image
            if args.mma in (None, 1) and not args.no_fast:
                eng.set_mma_mode(4)
                ms_fast = time_call(lambda: cycle_resident(lockstep=False), reps=1, warm=1)
                fast_img = cycle_resident(lockstep=False)
                um = time_call(lambda: unet(x2, t2, ctx2))
                eng.set_mma_mode(1 if args.mma is None else args.mma)
                extra['fast_path'] = {'mma_mode': 4, 'what': MMA_LABELS[4], 'images_per_s': round(B / (ms_fast / 1e3), 4),
                                      f'unet_ms_cfg_batch{2 * B}': round(um, 2), 'max_abs_delta_pixel_vs_faithful': float((fast_img - ref_img).abs().max()),
                                      'note': 'NOT a parity mode: reported separately, never the headline'}
            # HBM-bound kernels at the 64x64 level, timed alone (north_star: GroupNorm / fused ResBlock path vs HBM roofline)
            norm_probe = {}
            hh = LAT
            xg = torch.randn(2 * B, hh, hh, 320, device=d)
            gam, bet = torch.randn(320, device=d), torch.randn(320, device=d)
            ms = time_call(lambda: eng.op_groupnorm(xg, gam, bet, 1e-5, True), reps=10, warm=3)
            norm_probe['groupnorm_silu_stats_plus_apply'] = {'shape': list(xg.shape), 'ms': round(ms, 4),
                                                             'alg_gbs_1r1w': round(2 * 4 * xg.numel() / (ms * 1e-3) / 1e9, 1),
                                                             'moved_gbs_2r1w': round(3 * 4 * xg.numel() / (ms * 1e-3) / 1e9, 1)}
            xl = xg.view(-1, 320)
            ms = time_call(lambda: eng.op_layernorm(xl, gam, bet), reps=10, warm=3)
            norm_probe['layernorm'] = {'shape': list(xl.shape), 'ms': round(ms, 4), 'alg_gbs_1r1w': round(2 * 4 * xl.numel() / (ms * 1e-3) / 1e9, 1)}
            for v in norm_probe.values():
                v['frac_hbm'] = round(v['alg_gbs_1r1w'] / pk['hbm_gbs'], 4)
        else:
            t1 = torch.full((B,), 501., device=d)
            x1 = torch.randn(B, 3, RES, RES, device=d)
            unet_ms[f'batch{B}'] = round(time_call(lambda: src(x1, t1)), 2)
            families = family_report(eng, lambda: src(x1, t1), pk)
        roof = roofline_of(families, pk, value, cfg['tflop_per_image'], MMA_LABELS.get(args.mma, str(args.mma)))

    # the CPU leg is timed on rank 0 of the single-GPU run only (the other ranks would just wait at the closing barrier)
    cpu = cpu_baseline_sample(args.config, n_calls=3) if (rank == 0 and world == 1 and not args.no_cpu) else None

    if rank == 0:
        line = {
            'metric': cfg['metric'] + ' at 1/2/4/8 B200; ms/U-Net-call', 'value': round(value, 4), 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': round(ms_total / args.steps, 2), 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'fp32', 'data': 'synthetic (images U[0,1], conditioning N(0,1), random-init weights of the named topology)',
            'config': {'workload': cfg['name'], 'global_batch': world * B, 'steps_encode': S, 'steps_decode': S, 'eta': ETA,
                       'parallelism': f'dp{world} (images sharded, one NCCL weight broadcast)', 'mma_mode': MMA_LABELS.get(args.mma, str(args.mma)),
                       'l2': 'no flush: GBs of weights + >1 GB activations per U-Net call are streamed every call (>> 126 MB L2)',
                       'loop': ('lock-step: one U-Net call per step on [source | target uncond | target cond] (3B samples), recovered noise '
                                'consumed in the same step' if latent else 'two-phase: source-model encode, target-model decode'),
                       'unet_calls_per_step': (S if latent else 2 * S - 1), 'unet_ms': unet_ms, 'stage_ms_two_phase': stage_ms,
                       'launch': ('programmatic dependent launch (GEMM / attention / norm kernels)' if os.environ.get('CDX_PDL', '1') != '0'
                                  else 'stream-serialised launches (CDX_PDL=0)')},
            'e2e': {'value': round(e2e_value, 4), 'unit': UNIT, 'h2d_bytes_per_step': h2d[0], 'd2h_bytes_per_step': 4 * out_host.numel(),
                    'steps': e2e_steps, 'api': api},
            'gpu_launches': launches, 'clocks': clk, 'roofline': roof, 'kernel_families': families, 'hbm_bound_kernels': norm_probe,
            'cpu_baseline': cpu, 'weights_broadcast_ms': bcast_ms, 'setup_s': round(load_s, 1), 'workspace_gb': round(eng.workspace_bytes / 2 ** 30, 2),
        }
        line.update(extra)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ================================================================================================ CPU arms
def _host_threads():
    """CPU threads this process may really use: affinity mask, capped by the cgroup CPU quota (a container that shows
    128 CPUs but is throttled to a few cores thrashes with 128 ATen threads)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        with open('/sys/fs/cgroup/cpu.max') as fh:
            quota, period = fh.read().split()
        if quota != 'max':
            n = min(n, max(1, int(float(quota) / float(period) + 0.5)))
    except (OSError, ValueError):
        pass
    return max(1, min(n, 64))


_CPU_STATE = {}


def cpu_baseline_sample(config=2, n_calls=3):
    """The reference's CPU path (oracle port: same ATen CPU kernels, fp32) on a bounded sample of the same workload
    (BASELINE.md section 3): after one discarded cold call, `n_calls` (>= 3) warm U-Net forwards AT THE REAL LAUNCH BATCH of the
    encode loop (B) -- the CFG decode calls run at 2B and are counted as two such forwards -- plus (latent configs, once per process)
    one VAE encode + decode of one image.  images/s = B / (n_forwards_at_B * t_forward + B * t_vae)."""
    from cycle_diffusion_b200 import specs
    cfg = CONFIGS[config]
    st = _CPU_STATE.setdefault(config, {})
    B, S = cfg['B'], cfg['steps']
    if not st:
        st['threads'] = _host_threads()
        torch.set_num_threads(st['threads'])
        g = torch.Generator().manual_seed(0)
        if cfg['kind'] == 'latent':
            from oracle import unet_openai, vae_kl
            ucfg, vcfg = specs.sd_unet_config(cfg['ctx']), specs.kl_f8_config()
            usd = specs.synth_state_dict(specs.openai_unet_params(ucfg), 1234)
            vsd = specs.synth_state_dict(specs.kl_vae_params(vcfg), 1235)
            x = torch.randn(B, 4, cfg['lat'], cfg['lat'], generator=g)
            ctx = torch.randn(B, 77, cfg['ctx'], generator=g)
            img = torch.rand(1, 3, cfg['res'], cfg['res'], generator=g) * 2 - 1
            st['fwd'] = lambda: unet_openai.unet_forward(usd, ucfg, x, torch.full((B,), 501), ctx)
            with torch.no_grad():
                unet_openai.unet_forward(usd, ucfg, x[:1], torch.tensor([501]), ctx[:1])      # cold oneDNN call, discarded
                t0 = time.time()
                m = vae_kl.encode_moments(vsd, vcfg, img)
                vae_kl.decode(vsd, vcfg, m[:, :4])
                st['t_vae'] = time.time() - t0
            st['n_fwd'] = 3 * S                    # S encode calls at B + S CFG calls at 2B
        else:
            from oracle import unet_iddpm
            icfg = specs.iddpm_config(cfg['res'])
            sd = specs.synth_state_dict(specs.iddpm_unet_params(icfg), 1234)
            x = torch.randn(B, 3, cfg['res'], cfg['res'], generator=g)
            st['fwd'] = lambda: unet_iddpm.unet_forward(sd, icfg, x, torch.full((B,), 501.))
            with torch.no_grad():
                unet_iddpm.unet_forward(sd, icfg, x[:1], torch.tensor([501.]))
            st['t_vae'] = 0.0
            st['n_fwd'] = 2 * S - 1
    with torch.no_grad():
        t0 = time.time()
        for _ in range(n_calls):
            st['fwd']()
        t_fwd = (time.time() - t0) / n_calls
    value = B / (st['n_fwd'] * t_fwd + B * st['t_vae'])
    return {'value': round(value, 6), 'unit': UNIT, 'cores': st['threads'], 'kind': 'port',
            'sample': f'{n_calls} warm U-Net forwards at the real launch batch {B} ({t_fwd:.2f} s each)'
                      + (f' + VAE enc/dec of one {cfg["res"]}x{cfg["res"]} image ({st["t_vae"]:.2f} s)' if st['t_vae'] else '')
                      + f'; extrapolated: B / ({st["n_fwd"]} * t_forward + B * t_vae)',
            'unet_s_per_call_at_batch': round(t_fwd, 3), 'unet_batch': B, 'vae_s': round(st['t_vae'], 3)}


def run_reference(args):
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    vals = []
    t_all = time.time()
    for i in range(args.warmup + args.steps):
        r = cpu_baseline_sample(args.config, n_calls=1 if i < args.warmup else 3)
        if i >= args.warmup:
            vals.append(r)
        if time.time() - t_all > 200 and vals:   # keep the whole run within a few minutes
            break
    if not vals:
        vals = [r]
    v = sum(x['value'] for x in vals) / len(vals)
    cpu = dict(vals[-1])
    cpu['value'] = round(v, 6)
    line = {'impl': 'reference', 'metric': cfg['metric'] + ' at 1/2/4/8 B200; ms/U-Net-call', 'value': round(v, 6), 'unit': UNIT, 'n_gpus': args.gpus,
            'steps': len(vals), 'warmup': args.warmup, 'ms_per_step': round(1e3 * cfg['B'] / v, 1), 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'fp32', 'data': 'synthetic',
            'config': {'workload': cfg['name'] + ' -- CPU path on a bounded sample',
                       'note': 'the reference is Python and cannot travel to the GPU box; this is its CPU restatement (oracle/), same ATen kernels'},
            'cpu_baseline': cpu, 'e2e': {'value': round(v, 6), 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}, 'gpu_launches': 0}
    print(json.dumps(line))


def build_parser():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', type=int, default=2, choices=[2, 4, 5], help='BASELINE.json configuration (2 = configs[1], the headline)')
    ap.add_argument('--mma', type=int, default=None, help='0 FFMA fp32, 1 tcgen05 fp16-split (default), 3 tcgen05 3xTF32, 4 fast path')
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--no-fast', action='store_true', help='skip the fast-path probe')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help="write the images of the last timed step (rank 0's batch) to DIR/images.npy, float32")
    return ap


if __name__ == '__main__':
    ap = build_parser()
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)
