"""
CPU tests of bench.py's host-side pieces: the reference arm (`--impl reference`, the C/OpenMP port
of the reference on the host cores) prints one well-formed JSON line, and the bounded CPU-baseline
timers used by the `--op mi` / `--op blur` lines run.  (The GPU arm needs a device.)
"""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '2', '--warmup', '1'],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['unit'] == 'voxels/s' and d['higher_is_better'] is True
    assert d['value'] > 0 and d['steps'] == 2 and d['gpu_launches'] == 0 and d['warmup'] >= 3
    assert d['config']['batch_per_gpu'] == 8 and 'MEDIAN' in d['cpu_baseline']['sample']
    assert d['e2e']['value'] == d['value'] and d['e2e']['h2d_bytes_per_step'] == 0
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1
    assert '160x192x224' in d['metric'] and d['config']['volume'] == [160, 192, 224]


def test_cpu_legs_respect_the_container_cpu_quota(monkeypatch, tmp_path):
    """the GPU boxes show 128 cores but give the container 16 CPUs per period (cgroup v2 cpu.max): the CPU legs must not
    start more runnable threads than that (they get throttled into a bimodal timing); v1 files and 'max' are understood"""
    import builtins
    from oracle import cport
    real_open = builtins.open
    files = {}

    def fake_open(path, *a, **k):
        if isinstance(path, str) and path.startswith('/sys/fs/cgroup/'):
            if path not in files:
                raise FileNotFoundError(path)
            f = tmp_path / path.strip('/').replace('/', '_')
            f.write_text(files[path])
            return real_open(f, *a, **k)
        return real_open(path, *a, **k)

    monkeypatch.setattr(builtins, 'open', fake_open)
    files['/sys/fs/cgroup/cpu.max'] = '1600000 100000\n'
    assert cport.cgroup_cpu_limit() == 16.0
    monkeypatch.setattr(os, 'sched_getaffinity', lambda pid: set(range(128)))
    before = cport.num_threads()
    try:
        assert cport.use_all_cores() == 16
        files['/sys/fs/cgroup/cpu.max'] = 'max 100000\n'
        assert cport.cgroup_cpu_limit() is None
        del files['/sys/fs/cgroup/cpu.max']
        files['/sys/fs/cgroup/cpu/cpu.cfs_quota_us'] = '-1\n'
        files['/sys/fs/cgroup/cpu/cpu.cfs_period_us'] = '100000\n'
        assert cport.cgroup_cpu_limit() is None
        files['/sys/fs/cgroup/cpu/cpu.cfs_quota_us'] = '250000\n'
        assert cport.cgroup_cpu_limit() == 2.5
        assert cport.use_all_cores() == 2
    finally:
        cport.set_num_threads(before)


def test_bounded_cpu_baseline_timers():
    import bench
    from oracle import cport
    x = np.random.default_rng(0).uniform(0, 1, (1, 12, 14, 16, 1)).astype(np.float32)
    y = (x * x).astype(np.float32)
    r = bench.cpu_record(lambda: cport.mi_channelwise(x, y, nb_bins=16), x.size, 'voxels/s', 'tiny', budget_s=0.2, min_runs=5)
    assert r['value'] > 0 and r['unit'] == 'voxels/s' and r['kind'] == 'port' and r['cores'] >= 1 and 'median of' in r['sample']
    r = bench.cpu_record(lambda: cport.gaussian_blur(x, 1.0), x.size, 'voxels/s', 'tiny', budget_s=0.2, min_runs=5)
    assert r['value'] > 0
    # the statistic: median of the sorted run times, never fewer than min_runs runs
    calls = []
    med, n, best = bench.median_time(lambda: calls.append(1), budget_s=0.0, min_runs=7, warm=1)
    assert n == 7 and len(calls) == 8 and best <= med


def test_host_placement_helpers():
    import bench
    assert bench.parse_cpulist('0-3,8,10-11') == {0, 1, 2, 3, 8, 10, 11}
    assert bench.parse_cpulist('') == set()


def test_reference_arm_and_our_arm_share_one_config():
    """VERDICT r1: `same_config` was false because the reference arm's config lacked batch_per_gpu."""
    import argparse
    import bench
    a = argparse.Namespace(batch=8, flow='iid', method='linear')
    c = bench.warp_config(a, 1)
    assert c['batch_per_gpu'] == 8 and c['volume'] == [160, 192, 224] and 'configs[1]' in c['workload']


def test_dump_outputs_writes_the_last_step_and_a_fixed_sample_of_large_outputs(tmp_path):
    import argparse
    import torch
    import bench
    args = argparse.Namespace(dump_outputs=str(tmp_path / 'dump'))
    small = torch.arange(10, dtype=torch.float64)
    big = torch.arange(bench.DUMP_ELEMS + 1000, dtype=torch.float32).reshape(-1, 8)
    bench.dump_output(args, 'small', [small * 0, small])
    bench.dump_output(args, 'big', [big])
    bench.dump_output(args, 'big_again', [big.clone()])
    bench.dump_output(args, 'other_rank', [small], rank=1)
    s = np.load(tmp_path / 'dump' / 'small.npy')
    assert s.dtype == np.float32 and np.array_equal(s, np.arange(10))
    b = np.load(tmp_path / 'dump' / 'big.npy')
    assert b.dtype == np.float32 and b.shape == (bench.DUMP_ELEMS,) and np.all(np.diff(b) > 0)
    assert np.array_equal(b, np.load(tmp_path / 'dump' / 'big_again.npy'))
    assert not (tmp_path / 'dump' / 'other_rank.npy').exists()
    bench.dump_output(argparse.Namespace(dump_outputs=None), 'off', [small])
    assert sorted(os.listdir(tmp_path / 'dump')) == ['big.npy', 'big_again.npy', 'small.npy']


def test_timed_region_times_exactly_k_steps_and_hands_over_the_last_output(monkeypatch):
    import torch
    import bench
    calls = []

    class Event:
        def __init__(self, enable_timing=False):
            self.at = None

        def record(self):
            self.at = len(calls)

        def elapsed_time(self, end):
            return float(end.at - self.at)          # 1 ms per call between the two events

    monkeypatch.setattr(torch.cuda, 'Event', Event)
    monkeypatch.setattr(torch.cuda, 'synchronize', lambda *a: None)

    def fn():
        calls.append(1)
        return len(calls)
    for steps, warmup in ((7, 5), (1, 0), (0, 4)):
        calls.clear()
        last = []
        ms = bench.timed_region(fn, steps, warmup, 1, min_preheat_s=0.0, last=last)
        assert ms == steps and len(calls) == max(warmup, 3) + steps
        assert last == ([len(calls)] if steps else [])


def test_step_flags_set_the_steps_of_every_record(monkeypatch, capsys):
    import argparse
    import torch
    import bench
    seen = {}

    def fake(name):
        def rec(args, world, rank, dev, steps, *a, **k):
            key = name + ('_cce' if k.get('cce') else '') + ('_b%d' % k['batch'] if k.get('batch') else '')
            seen[key] = steps
            return {'config': {'workload': key}, 'metric': key, 'value': 1.0, 'unit': 'u', 'steps': steps,
                    'ms_per_step': 1.0, 'gpu_launches': steps,
                    'roofline': dict.fromkeys(('achieved', 'peak', 'frac', 'bytes_model', 'traffic', 'traffic_source'))}
        return rec
    for name in ('dice', 'lc3d', 'resize', 'warp_mc', 'slab', 'cfg5'):
        monkeypatch.setattr(bench, name + '_record', fake(name))
    # the default line's sub-records follow --long-steps
    bench.run_ops(argparse.Namespace(long_steps=13), 1, 0, 0, torch.device('cpu'))
    assert seen == {'dice': 13, 'dice_cce': 13, 'lc3d_b1': 13, 'lc3d_b8': 13, 'resize': 13, 'warp_mc': 13}
    # an --op line times --steps (cfg5: --cfg5-steps)
    monkeypatch.setattr(torch.cuda, 'is_available', lambda: True)
    monkeypatch.setattr(bench, 'dist_setup', lambda n: (1, 0, 0))
    for op, key in (('dice', 'dice'), ('cce', 'dice_cce'), ('lc3d', 'lc3d'), ('resize', 'resize'), ('warp_mc', 'warp_mc'),
                    ('warp_slab', 'slab_b1'), ('cfg5', 'cfg5')):
        seen.clear()
        monkeypatch.setattr(sys, 'argv', ['bench.py', '--op', op, '--steps', '7', '--cfg5-steps', '4'])
        bench.main()
        assert seen == {key: 4 if op == 'cfg5' else 7}
        assert json.loads(capsys.readouterr().out.strip().splitlines()[-1])['steps'] == seen[key]


def test_gpu_arm_refuses_to_run_without_a_device():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '1', '--warmup', '1'],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0 and 'no CUDA device' in (out.stderr + out.stdout)
