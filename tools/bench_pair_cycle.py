"""Two-model pixel translation: two-phase (source.encode -> z -> target(z)) against the lock-step loop (source.pair_cycle(target)),
alternated in one process on the same inputs and seeds.

Workloads (two i-DDPM 256x256 U-Nets with random-init weights, each on its own engine as UnsupervisedTranslation builds them,
DDIM eta 0.1, rng='cuda'):
  cfg5  bench.py --config 5's shape: 250 steps, es_steps 250, B = 8
  afhq  the paper's AFHQ cat -> dog settings at B = 1: custom_steps 1000, es_steps 850, refine_steps 100
        (translate_afhqcat256_to_afhqdog256_ddim_eta01.cfg); --es-steps shortens it for a rehearsal

Per mode and repetition: ms per image from CUDA events after a synchronise, kernel launches (both engines), peak
torch.cuda.max_memory_allocated plus the engines' workspace bytes; per workload: torch.equal of the two outputs and the spread
of the repetitions.  The GPU name and power limit are read in the same run.  One JSON document goes to stdout (and --out).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    info = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30)
        info['power_limit_and_max_sm_clock'] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as err:
        info['power_limit_and_max_sm_clock'] = f'not read: {err}'
    return info


def build(workload, es_override):
    from cycle_diffusion_b200 import specs
    from cycle_diffusion_b200.engine import Engine, UNet
    from cycle_diffusion_b200.wrappers import DDPMDDIMWrapper
    if workload == 'cfg5':
        B, kw = 8, dict(sample_type='ddim', eta=0.1, custom_steps=250, es_steps=250)
    else:
        B, kw = 1, dict(sample_type='ddim', eta=0.1, custom_steps=1000, es_steps=es_override or 850, refine_steps=100)
    eng = Engine(0)
    eng2 = Engine(0)
    cfg = specs.iddpm_config(256)
    src = UNet(eng, cfg, 'iddpm').load_state_dict(specs.synth_state_dict(specs.iddpm_unet_params(cfg), 1234))
    tgt = UNet(eng2, cfg, 'iddpm').load_state_dict(specs.synth_state_dict(specs.iddpm_unet_params(cfg), 4321))
    w_src = DDPMDDIMWrapper('cat256', unet=src, image_size=256, rng='cuda', **kw)
    w_tgt = DDPMDDIMWrapper('dog256', unet=tgt, image_size=256, rng='cuda', **kw)
    assert w_src.pair_cycle_applies(w_tgt)
    image = torch.rand(B, 3, 256, 256, generator=torch.Generator().manual_seed(0)).to(eng.device)
    engines = [eng, eng2]
    return B, kw, w_src, w_tgt, image, engines


def run_mode(mode, w_src, w_tgt, image, engines, seed=99):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    l0 = sum(e.launches for e in engines)
    torch.manual_seed(seed)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    if mode == 'lockstep':
        out = w_src.pair_cycle(w_tgt, image)
    else:
        out = w_tgt(w_src.encode(image))
    b.record()
    torch.cuda.synchronize()
    return out, dict(ms=a.elapsed_time(b), launches=sum(e.launches for e in engines) - l0,
                     peak_torch_bytes=torch.cuda.max_memory_allocated(), workspace_bytes=sum(e.workspace_bytes for e in engines))


def bench(workload, reps, es_override):
    B, kw, w_src, w_tgt, image, engines = build(workload, es_override)
    modes = ('two_phase', 'lockstep')
    outs = {}
    for m in modes:                                    # warm-up: module loads, workspace growth
        outs[m] = run_mode(m, w_src, w_tgt, image, engines)[0]
    runs = {m: [] for m in modes}
    for r in range(reps):
        for m in (modes if r % 2 == 0 else modes[::-1]):
            out, rec = run_mode(m, w_src, w_tgt, image, engines)
            runs[m].append(rec)
            outs[m] = out
    res = dict(workload=workload, batch=B, schedule=kw, z_bytes=B * kw['es_steps'] * 3 * 256 * 256 * 4,
               outputs_equal=bool(torch.equal(outs['two_phase'], outs['lockstep'])))
    for m in modes:
        ms_img = [x['ms'] / B for x in runs[m]]
        res[m] = dict(ms_per_image=[round(v, 2) for v in ms_img], ms_per_image_median=round(statistics.median(ms_img), 2),
                      spread_pct=round(100 * (max(ms_img) - min(ms_img)) / statistics.median(ms_img), 2),
                      launches=runs[m][-1]['launches'],
                      peak_bytes=max(x['peak_torch_bytes'] for x in runs[m]) + runs[m][-1]['workspace_bytes'],
                      peak_torch_bytes=max(x['peak_torch_bytes'] for x in runs[m]), workspace_bytes=runs[m][-1]['workspace_bytes'])
    res['lockstep_vs_two_phase_time'] = round(res['lockstep']['ms_per_image_median'] / res['two_phase']['ms_per_image_median'], 4)
    return res


def main():
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument('--workload', choices=['cfg5', 'afhq', 'both'], default='both')
    p.add_argument('--reps', type=int, default=3)
    p.add_argument('--es-steps', type=int, default=None, help='afhq: shorten es_steps (rehearsal)')
    p.add_argument('--out', default=None, help='also write the JSON document here')
    a = p.parse_args()
    if not torch.cuda.is_available():
        sys.exit('bench_pair_cycle: needs a CUDA device (there is no CPU measurement)')
    doc = dict(gpu=gpu_info(), reps=a.reps, results=[])
    for w in (['cfg5', 'afhq'] if a.workload == 'both' else [a.workload]):
        doc['results'].append(bench(w, a.reps, a.es_steps))
        print(json.dumps(doc['results'][-1]), file=sys.stderr, flush=True)
    txt = json.dumps(doc, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(txt)


if __name__ == '__main__':
    main()
