"""bench.py: the output contract checked on a LIVE run (GPU) and the host-side helpers (CPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

REQUIRED = ['metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline', 'dtype',
            'data', 'config', 'e2e', 'gpu_launches', 'clocks', 'roofline', 'cpu_baseline']


def test_defaults_are_the_single_gpu_headline():
    import bench
    ap = bench.build_parser()
    a = ap.parse_args([])
    assert a.gpus == 1 and a.config == 2 and a.warmup >= 3 and a.impl == 'ours' and a.dump_outputs is None


def test_host_thread_budget_is_sane():
    import bench
    n = bench._host_threads()
    assert 1 <= n <= 64 and n <= (os.cpu_count() or 1)


def test_bench_never_routes_the_product_through_the_oracle():
    """Only the CPU legs may touch oracle/: the import sits inside the two CPU-arm functions."""
    src = open(os.path.join(ROOT, 'bench.py')).read()
    head = src.split('# ================================================================================================ CPU arms')[0]
    assert 'import oracle' not in head and 'from oracle' not in head


@pytest.mark.gpu
def test_live_bench_line_has_the_contract_keys(tmp_path):
    """One short real run (LDM 256^2 configuration, 1 timed step, no CPU leg): every contract key, consistent bookkeeping, and the
    images of the timed step written by --dump-outputs."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--config', '4', '--steps', '1', '--warmup', '3', '--no-cpu', '--no-fast',
                        '--dump-outputs', str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    for k in REQUIRED:
        assert k in d, k
    assert d['higher_is_better'] is True and d['scaling'] == 'weak' and d['vs_baseline'] is None and d['n_gpus'] == 1
    assert 'workload' in d['config'] and 'model' not in d['config']
    assert set(['value', 'unit', 'h2d_bytes_per_step', 'd2h_bytes_per_step']) <= set(d['e2e'])
    assert d['e2e']['h2d_bytes_per_step'] > 0 and d['e2e']['d2h_bytes_per_step'] > 0 and d['e2e']['value'] > 0
    assert d['gpu_launches'] > 0
    ro = d['roofline']
    assert ro['bound'] in ('hbm', 'tensor') and abs(ro['frac'] - ro['achieved'] / ro['peak']) < 1e-3 and 0 < ro['frac'] < 1.2
    assert not (set(d['clocks']['reasons']) & {'hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown'})
    # throughput bookkeeping: value = images per step / seconds per step; e2e cannot beat the resident number by much
    assert abs(d['value'] - d['config']['global_batch'] / (d['ms_per_step'] / 1e3)) < 1e-2 * d['value'] + 1e-3
    assert d['e2e']['value'] < 1.1 * d['value']
    # the two loop drivers agree
    assert d['two_phase']['max_abs_diff_lockstep_vs_two_phase'] < 1e-3
    assert sorted(os.listdir(tmp_path)) == ['images.npy']
    img = np.load(tmp_path / 'images.npy')
    assert img.dtype == np.float32 and img.shape == (d['config']['global_batch'], 3, 256, 256) and np.isfinite(img).all()
