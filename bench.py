#!/usr/bin/env python
"""
bench.py -- BASELINE.json's metric: voxels/s warped (SpatialTransformer / interpn linear) on
160x192x224 fp32 volumes, with the achieved fraction of the HBM roofline.

    python bench.py --gpus 1 --steps K --warmup W                 # our CUDA path
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...                           # CPU port of the reference, host cores
    python bench.py --op dice|cce|lc3d|resize|warp_mc|warp_slab|cfg5|mi|mi_segs|blur ...   # one op per line
    python bench.py ... --dump-outputs DIR                         # + DIR/<name>.npy: the last timed step's output

The inputs are drawn from fixed seeds, so two builds run with the same arguments can be compared output for output
through --dump-outputs.  Every record that runs a timed step writes one array: the headline warp as warp.npy, the
default line's ops as dice, cce, lc3d, lc3d_b8, resize and warp_c16, its N-GPU records as slab, slab_c16, cfg5_batch and
cfg5_slab, and the --op lines under their own names (mi, mi_segs, blur, slab / slab_c<C>, lc3d_b<B>, warp_c<C>, ...).
At N GPUs, rank 0 writes what it computed: its own batch, or its planes of a z-slab-sharded volume.  --impl reference
runs no GPU step and writes nothing.

Step counts: --steps sets the timed steps of the line's own measurement, --long-steps those of the headline's long_run
and of every sub-record of the default line, --e2e-steps and --cfg5-steps those of the e2e and cfg5 records.

A "step" is one pass of the hot path over one batch: `--batch` (default 8) independent
160x192x224x1 volumes with a random dense 3-channel flow U(-3,3) (configs[1] of
BASELINE.json, SURVEY.md 8d), one kernel launch.  The batch's working set is 1.1 GB, far
larger than the 126 MB L2, so no flush is needed between iterations.  At N GPUs every rank
warps its own batch (weak scaling, no data-path collective); `value` is whole-job
voxels/s = N * batch * V * K / max-over-ranks device time (CUDA events, barrier + sync on
both sides).

JSON keys beyond the base contract:
  roofline     achieved = 20 B/voxel (12 flow + 4 source-once + 4 store, SURVEY.md 8d)
               * voxels per launch / launch time; peak = MEASURED_PEAKS.json hbm_gbs.
               `traffic` is the ncu dram__bytes of the committed capture (profiles/traffic.json, static).
  long_run     the same launch timed over --long-steps steps (default 200; K steps of a short run are only a few ms)
  e2e          the same metric through the public API with HOST (pinned) buffers: H2D of
               vol+flow and D2H of the result inside the timed region, every step.
  cpu_baseline the oracle's C/OpenMP port on the host cores, bounded sample (rank 0, N=1), MEDIAN of >= 20 runs
               with bound threads and first-touched inputs -- the same recipe as --impl reference.
  ops          (N = 1) the other BASELINE.json configs, each with ms_per_step, roofline and its own cpu_baseline:
               Dice, CCE (configs[2]), LocallyConnected3D (configs[3]), Resize, 16-channel warp (configs[4]'s kernel)
  slab         (N > 1) ONE 160x192x224 volume sharded in z-slabs over the N ranks with the halo exchange
               (strong scaling): overlapped plan vs serial path, exchange-only and kernels-only times
  cfg5         (N > 1) BASELINE.json configs[4]: UNet fwd -> 16-channel warp -> Dice, batch-sharded and z-slab-sharded
"""
import argparse
import importlib.util
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SHAPE = (160, 192, 224)
V = SHAPE[0] * SHAPE[1] * SHAPE[2]


def measured_peak():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    except Exception:                                       # noqa: BLE001
        return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


def ncu_traffic(op):
    """dram bytes per launch from the committed ncu summary, if present (profiles/traffic.json): a STATIC number
    taken from the capture under profiles/, not a measurement of this run."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'traffic.json')) as f:
            return json.load(f).get(op)
    except Exception:                                       # noqa: BLE001
        return None


def roofline(nbytes_per_step, ms_per_step, traffic_key, model, kernel=None):
    peak, peak_src = measured_peak()
    achieved = nbytes_per_step / (ms_per_step * 1e-3) / 1e9
    r = {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
         'traffic': ncu_traffic(traffic_key), 'traffic_source': 'profiles/traffic.json (static, from the committed ncu capture)',
         'peak_source': peak_src, 'bytes_model': model, 'per': 'GPU'}
    if kernel:
        r['kernel'] = kernel
    return r


class ClockSampler:
    """Samples SM clock / throttle reasons through NVML while the benchmark runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:                                   # noqa: BLE001
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {'hw_slowdown': 0x8, 'sw_power_cap': 0x4, 'sw_thermal_slowdown': 0x20,
                 'hw_thermal_slowdown': 0x40, 'hw_power_brake': 0x80}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:                               # noqa: BLE001
                pass
            time.sleep(0.01)

    def start(self):
        if self.nv:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
        return self

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join()
        s = sorted(self.samples)
        return {'sm_mhz': s[len(s) // 2] if s else None, 'sm_max_mhz': self.max_mhz,
                'reasons': sorted(self.reasons), 'samples': len(s)}


# ---------------------------------------------------------------------------------------
# host placement: one rank per GPU, its thread and pinned buffers on the GPU's NUMA node
# ---------------------------------------------------------------------------------------
def gpu_numa_cpus(index):
    """CPUs of the NUMA node the GPU hangs off (sysfs), or None if the topology is not exposed."""
    try:
        import torch
        p = torch.cuda.get_device_properties(index)
        bdf = '%04x:%02x:%02x.0' % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        with open('/sys/bus/pci/devices/%s/numa_node' % bdf) as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open('/sys/devices/system/node/node%d/cpulist' % node) as f:
            return parse_cpulist(f.read().strip()), node
    except Exception:                                       # noqa: BLE001
        return None


def parse_cpulist(s):
    cpus = set()
    for part in s.split(','):
        part = part.strip()
        if not part:
            continue
        if '-' in part:
            a, b = part.split('-')
            cpus.update(range(int(a), int(b) + 1))
        else:
            cpus.add(int(part))
    return cpus


def bind_host_to_gpu(local):
    """Pin this process to the CPUs of its GPU's NUMA node BEFORE any pinned buffer is allocated, so that the
    staging memory of the end-to-end path is first-touched next to the PCIe root it is copied through (8 ranks
    on a 2-socket box otherwise all allocate on whichever node the launcher started them).  Returns a note for
    the JSON line; the original mask is kept for the CPU-baseline leg (which uses every core)."""
    try:
        orig = os.sched_getaffinity(0)
    except AttributeError:
        return None, {'numa': 'unsupported platform'}
    found = gpu_numa_cpus(local)
    if not found:
        return orig, {'numa': 'topology not exposed; affinity unchanged'}
    cpus, node = found
    cpus = (cpus & orig) or cpus
    try:
        os.sched_setaffinity(0, cpus)
    except OSError as ex:
        return orig, {'numa': 'sched_setaffinity failed: %s' % ex}
    return orig, {'numa_node': node, 'cpus_bound': len(cpus)}


def dist_setup(n_gpus):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        import datetime
        # a short collective timeout: a rank that fails must not leave the others (and the driver) hanging for the
        # default 10 minutes
        dist.init_process_group('nccl', device_id=torch.device('cuda', local), timeout=datetime.timedelta(seconds=180))
    return world, rank, local


def timed_region(fn, steps, warmup, world, min_preheat_s=0.3, last=None):
    """W warm-up steps, then exactly K steps between CUDA events, barrier + sync both sides,
    max over ranks.  A short pre-heat (not counted) lets the clocks settle and gives the
    sampler something to see.  If `last` is a list, what the K-th timed call returned is appended to it."""
    import torch
    import torch.distributed as dist
    if world > 1:
        # a FIXED number of pre-heat calls: `fn` may contain collectives, so every rank must call it equally often
        for _ in range(10 if min_preheat_s > 0 else 0):
            fn()
        torch.cuda.synchronize()
    else:
        t0 = time.time()
        while time.time() - t0 < min_preheat_s:
            fn()
            torch.cuda.synchronize()
    for _ in range(max(warmup, 3)):
        fn()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        dist.barrier()
        t = torch.tensor([ms], dtype=torch.float64, device='cuda')
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    if last is not None and steps > 0:
        last.append(out)
    return float(ms)


DUMP_ELEMS = 1 << 21          # 8 MB of float32 per array; a line dumps at most 7 arrays, under 64 MB in all


def dump_output(args, name, last, rank=0):
    """--dump-outputs DIR: what the last timed step returned, as DIR/<name>.npy in float32.  An output of more than
    DUMP_ELEMS elements is sampled at DUMP_ELEMS flat indices drawn from a fixed seed, the same in every run."""
    if not args.dump_outputs or rank != 0:
        return
    import numpy as np
    import torch
    out = last[-1].detach().reshape(-1)
    if out.numel() > DUMP_ELEMS:
        idx = np.sort(np.random.default_rng(0).choice(out.numel(), DUMP_ELEMS, replace=False))
        out = out[torch.from_numpy(idx).to(out.device)]
    os.makedirs(args.dump_outputs, exist_ok=True)
    np.save(os.path.join(args.dump_outputs, name + '.npy'), out.float().cpu().numpy())


# ---------------------------------------------------------------------------------------
# CPU arm: the oracle's C/OpenMP port, bound threads, first-touched inputs, median
# ---------------------------------------------------------------------------------------
_CPU_READY = False


def cpu_setup(orig_affinity=None):
    """One recipe for BOTH CPU legs (cpu_baseline of our arm and --impl reference): threads bound to cores
    (OMP_PROC_BIND=close, OMP_PLACES=cores -- must be in the environment before libgomp starts), as many threads as
    the box gives this container -- min(cores in the affinity mask, cgroup CPU quota): the GPU boxes show 128 cores
    but cap the container at 16 CPUs per 100 ms period, and 128 runnable threads get the whole group throttled for
    the rest of a period (tools/cpu_leg_probe.py: 4.5 ms best, 94 ms median with 128 threads; 20.4-20.8 ms min-max
    with 16) -- inputs first-touched by the OpenMP threads, the MEDIAN of >= 20 runs reported."""
    global _CPU_READY
    if orig_affinity:
        try:
            os.sched_setaffinity(0, orig_affinity)
        except OSError:
            pass
    if not _CPU_READY:
        os.environ.setdefault('OMP_PROC_BIND', 'close')
        os.environ.setdefault('OMP_PLACES', 'cores')
        # passive: idle OpenMP threads must not keep spinning into the container's CPU quota while the GPU legs run
        os.environ.setdefault('OMP_WAIT_POLICY', 'passive')
        from oracle import cport
        cport.build()
        cport.use_all_cores()
        _CPU_READY = True
    from oracle import cport
    return cport


def median_time(fn, budget_s=6.0, min_runs=20, max_runs=200, warm=2):
    for _ in range(warm):
        fn()
    ts, t_all = [], time.time()
    while len(ts) < min_runs or (time.time() - t_all < budget_s and len(ts) < max_runs):
        t = time.time()
        fn()
        ts.append(time.time() - t)
    ts.sort()
    return ts[len(ts) // 2], len(ts), ts[0]


def cpu_record(fn, units, unit, what, budget_s=6.0, min_runs=20):
    cport = cpu_setup()
    med, n, best = median_time(fn, budget_s, min_runs)
    return {'value': units / med, 'unit': unit, 'cores': cport.num_threads(), 'kind': 'port',
            'cgroup_cpu_limit': cport.cgroup_cpu_limit(),
            'sample': '%s; median of %d runs (best %.3g %s), threads bound (OMP_PROC_BIND=close, OMP_PLACES=cores), '
                      'inputs first-touched by the OpenMP threads' % (what, n, units / best, unit)}


def synth_host_volume(seed=0):
    import numpy as np
    vol = np.random.default_rng(seed).standard_normal((1,) + SHAPE + (1,)).astype(np.float32)
    flow = np.random.default_rng(seed + 1).uniform(-3, 3, (1,) + SHAPE + (3,)).astype(np.float32)
    return vol, flow


def cpu_warp_callable(method):
    import numpy as np
    cport = cpu_setup()
    vol, flow = synth_host_volume()
    vol, flow = cport.first_touch(vol), cport.first_touch(flow)
    out = cport.first_touch(np.zeros(vol.shape, dtype=np.float32))
    return lambda: cport.warp(vol, flow, method, out=out)


def cpu_baseline_warp(method, budget_s=6.0):
    """The oracle's C/OpenMP port (same arithmetic as the reference, fused, all host threads)."""
    return cpu_record(cpu_warp_callable(method), V, 'voxels/s',
                      'oracle/c (C99+OpenMP restatement of interpn, -ffp-contract=off), ONE 160x192x224 volume per run',
                      budget_s)


def cpu_baseline_warp_numpy(method):
    """op-for-op numpy restatement (mirrors the reference's unfused TF op sequence), 1 thread."""
    from oracle import interp
    vol, flow = synth_host_volume()
    t = time.time()
    interp.spatial_transformer(vol, flow, method)
    dt = time.time() - t
    return {'value': V / dt, 'unit': 'voxels/s', 'cores': 1, 'kind': 'port',
            'sample': 'oracle/interp.py (numpy, op-for-op like the reference TF graph), one 160x192x224 volume, 1 run'}


def warp_workload(batch, flow='iid'):
    return ('SpatialTransformer warp of 160x192x224x1 fp32 volumes, random dense 3-ch flow (%s), batch %d per GPU per step '
            '(BASELINE.json configs[1])' % ('U(-3,3) i.i.d.' if flow == 'iid' else 'smooth, max|u|=8', batch))


def warp_config(args, world=1):
    return {'workload': warp_workload(args.batch, args.flow), 'batch_per_gpu': args.batch, 'volume': list(SHAPE),
            'channels': 1, 'interp_method': args.method,
            'parallelism': 'batch-sharded x%d, no collective' % world,
            'l2': 'working set %.2f GB per step > 126 MB L2 (no flush needed)' % (20.0 * args.batch * V / 1e9)}


def bench_reference(args):
    """--impl reference: the reference's CPU path (its C/OpenMP port; TensorFlow is not
    installable here, see DESIGN.md) on the host cores.  Rank 0 only.  Same recipe and statistic as the
    cpu_baseline leg of our arm (cpu_setup / median)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    world = int(os.environ.get('WORLD_SIZE', '1'))
    cport = cpu_setup()
    fn = cpu_warp_callable(args.method)
    warm = max(args.warmup, 3)
    for _ in range(warm):
        fn()
    steps = args.steps
    ts = []
    for _ in range(steps):
        t = time.time()
        fn()
        ts.append(time.time() - t)
    ts.sort()
    med = ts[len(ts) // 2]
    value = V / med
    sample = ('each step = ONE 160x192x224 volume (bounded sample of the batch-%d step), oracle/c C99+OpenMP port, '
              '%d threads bound to cores, inputs first-touched by the OpenMP threads; value = V / MEDIAN step time over the '
              '%d steps (best %.3g, worst %.3g voxels/s)'
              % (args.batch, cport.num_threads(), steps, V / ts[0], V / ts[-1]))
    print(json.dumps({
        'impl': 'reference',
        'metric': 'voxels/s warped (SpatialTransformer / interpn %s), 160x192x224 fp32' % args.method,
        'value': value, 'unit': 'voxels/s', 'n_gpus': world, 'steps': steps,
        'warmup': warm, 'ms_per_step': med * 1e3, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': warp_config(args, world),
        'cpu_baseline': {'value': value, 'unit': 'voxels/s', 'cores': cport.num_threads(), 'kind': 'port',
                         'cgroup_cpu_limit': cport.cgroup_cpu_limit(), 'sample': sample},
        'e2e': {'value': value, 'unit': 'voxels/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }), flush=True)


# ---------------------------------------------------------------------------------------
# the headline: BASELINE.json configs[1]
# ---------------------------------------------------------------------------------------
def bench_warp(args):
    import torch
    import neurite_b200 as ne
    world, rank, local = dist_setup(args.gpus)
    orig_aff, numa_note = bind_host_to_gpu(local)
    dev = torch.device('cuda', local)
    B = args.batch
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    vol = torch.randn((B,) + SHAPE + (1,), device=dev, generator=g)
    flow = torch.rand((B,) + SHAPE + (3,), device=dev, generator=g) * 6 - 3
    if args.flow == 'smooth':
        # low-frequency field, max |u| = 8 voxels (SURVEY.md 8d secondary run)
        coarse = torch.randn((B, 3, 10, 12, 14), device=dev, generator=g)
        flow = torch.nn.functional.interpolate(coarse, size=SHAPE, mode='trilinear', align_corners=True)
        flow = (flow / flow.abs().amax() * 8).permute(0, 2, 3, 4, 1).contiguous()
    st = ne.layers.SpatialTransformer(interp_method=args.method, fill_value=None, halo=args.halo)
    sampler = ClockSampler(local).start()
    last = []
    ms = timed_region(lambda: st([vol, flow]), args.steps, args.warmup, world, last=last)
    long_steps = args.long_steps
    ms_long = timed_region(lambda: st([vol, flow]), long_steps, 3, world, min_preheat_s=0.0)
    clocks = sampler.stop()
    vox_per_step = world * B * V
    value = vox_per_step * args.steps / (ms * 1e-3)
    bytes_per_launch = 20.0 * B * V

    # ---- end to end through the public API with host buffers (pinned, allocated after the NUMA binding)
    e2e_steps = args.e2e_steps
    h_vol = torch.empty(vol.shape, dtype=torch.float32).pin_memory().copy_(vol.cpu())
    h_flow = torch.empty(flow.shape, dtype=torch.float32).pin_memory().copy_(flow.cpu())
    h_out = torch.empty(vol.shape, dtype=torch.float32).pin_memory()

    def e2e_step():
        # public host-facing call: pinned host tensors in, pinned host tensor out; returns
        # only when the result is in h_out (H2D of vol+flow and D2H of the result inside)
        st.call_host([h_vol, h_flow], out=h_out)
    ms_e2e = timed_region(e2e_step, e2e_steps, 2, world, min_preheat_s=0.0)
    e2e_value = vox_per_step * e2e_steps / (ms_e2e * 1e-3)
    del h_vol, h_flow, h_out

    line = {
        'metric': 'voxels/s warped (SpatialTransformer / interpn %s), 160x192x224 fp32' % args.method,
        'value': value, 'unit': 'voxels/s', 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
        'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': warp_config(args, world),
        'roofline': roofline(bytes_per_launch, ms / args.steps, 'warp',
                             '20 B/voxel = 12 flow + 4 source (each voxel once) + 4 store', 'warp3d_tile_kernel'),
        'long_run': {'steps': long_steps, 'ms_per_step': ms_long / long_steps,
                     'value': vox_per_step * long_steps / (ms_long * 1e-3),
                     'roofline_frac': bytes_per_launch / (ms_long / long_steps * 1e-3) / 1e9 / measured_peak()[0],
                     'timed_region_s': ms_long * 1e-3},
        'e2e': {'value': e2e_value, 'unit': 'voxels/s', 'h2d_bytes_per_step': int(vol.numel() + flow.numel()) * 4,
                'd2h_bytes_per_step': int(vol.numel()) * 4, 'steps': e2e_steps, 'ms_per_step': ms_e2e / e2e_steps,
                'host_placement': numa_note},
        'gpu_launches': args.steps,
        'clocks': clocks,
    }
    # written after every timed region of the headline, so that the copy-out cannot disturb them
    dump_output(args, 'warp', last, rank)
    del vol, flow, last
    torch.cuda.empty_cache()
    # the NUMA binding was for the pinned staging buffers of the end-to-end path; the CPU legs below use every core
    if orig_aff:
        try:
            os.sched_setaffinity(0, orig_aff)
        except OSError:
            pass
    if not args.no_extras:
        if world == 1:
            line['ops'] = run_ops(args, world, rank, local, dev)
        else:
            for key, fn in (('slab', lambda: slab_record(args, world, rank, dev, args.long_steps, channels=1, batch=1)),
                            ('slab_c16', lambda: slab_record(args, world, rank, dev, args.long_steps, channels=16, batch=1)),
                            ('cfg5', lambda: cfg5_record(args, world, rank, dev, args.cfg5_steps))):
                try:
                    line[key] = fn()
                except Exception as ex:                      # noqa: BLE001 -- a sub-record must not take the headline down
                    line[key] = {'error': '%s: %s' % (type(ex).__name__, str(ex)[:300])}
                torch.cuda.empty_cache()
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            line['cpu_baseline'] = cpu_baseline_warp(args.method)
            if not args.no_numpy_baseline:
                line['cpu_baseline_numpy'] = cpu_baseline_warp_numpy(args.method)
        print(json.dumps(line), flush=True)
    finish(world)


def run_ops(args, world, rank, local, dev):
    """The other BASELINE.json configs inside the default line (driver-visible): compact records."""
    ops = {}
    steps = args.long_steps
    for name, fn in (('dice', lambda: dice_record(args, world, rank, dev, steps, cce=False)),
                     ('cce', lambda: dice_record(args, world, rank, dev, steps, cce=True)),
                     ('lc3d', lambda: lc3d_record(args, world, rank, dev, steps, batch=1)),
                     ('lc3d_b8', lambda: lc3d_record(args, world, rank, dev, steps, batch=8, cpu=False)),
                     ('resize', lambda: resize_record(args, world, rank, dev, steps)),
                     ('warp_c16', lambda: warp_mc_record(args, world, rank, dev, steps, 16))):
        try:
            r = fn()
            ops[name] = {'workload': r['config']['workload'], 'metric': r['metric'], 'value': r['value'], 'unit': r['unit'],
                         'steps': r['steps'], 'ms_per_step': r['ms_per_step'],
                         'roofline': {k: r['roofline'][k] for k in ('achieved', 'peak', 'frac', 'bytes_model', 'traffic', 'traffic_source')},
                         'gpu_launches': r['gpu_launches'], 'clocks': r.get('clocks'), 'cpu_baseline': r.get('cpu_baseline')}
        except Exception as ex:                              # noqa: BLE001 -- one op must not take the headline down
            ops[name] = {'error': '%s: %s' % (type(ex).__name__, str(ex)[:300])}
        import torch
        torch.cuda.empty_cache()
    return ops


# ---------------------------------------------------------------------------------------
# the other configs (own lines under --op; same timing discipline)
# ---------------------------------------------------------------------------------------
def base_line(metric, value, unit, world, steps, warmup, ms, scaling, workload, extra_cfg=None):
    cfg = {'workload': workload}
    cfg.update(extra_cfg or {})
    return {'metric': metric, 'value': value, 'unit': unit, 'n_gpus': world, 'steps': steps, 'warmup': max(warmup, 3),
            'ms_per_step': ms / steps, 'higher_is_better': True, 'scaling': scaling, 'vs_baseline': None, 'dtype': 'f32',
            'data': 'synthetic', 'config': cfg}


def dice_record(args, world, rank, dev, steps, cce=False):
    import numpy as np
    import torch
    import neurite_b200 as ne
    from neurite_b200.dist import slab_bounds
    B, L = 4, 16
    # cfg 3: batch 4 < 8 GPUs -> shard the voxel range of every batch item across ranks (strong scaling)
    z0, nz = slab_bounds(SHAPE[0], world, rank)
    g = torch.Generator(device=dev).manual_seed(7 + rank)
    lab = torch.randint(0, L, (B, nz) + SHAPE[1:], device=dev, generator=g)
    t = torch.nn.functional.one_hot(lab, L).float()
    p = torch.softmax(torch.randn((B, nz) + SHAPE[1:] + (L,), device=dev, generator=g), -1)
    group = torch.distributed.group.WORLD if world > 1 else None
    op = ne.losses.CategoricalCrossentropy(group=group) if cce else ne.losses.Dice(group=group)
    sampler = ClockSampler(dev.index).start()
    last = []
    ms = timed_region(lambda: op.loss(t, p), steps, args.warmup, world, last=last)
    clocks = sampler.stop()
    dump_output(args, 'cce' if cce else 'dice', last, rank)
    elems = B * V * L
    name = 'CategoricalCrossentropy' if cce else 'Dice().loss'
    line = base_line('(voxel,label) elements/s, %s on 16-label one-hot 160x192x224, batch 4' % ('CCE' if cce else 'Dice loss'),
                     elems * steps / (ms * 1e-3), 'elements/s', world, steps, args.warmup, ms, 'strong',
                     'BASELINE.json configs[2]: %s, y_true one-hot / y_pred softmax [4,160,192,224,16], voxel range sharded '
                     'over %d GPU(s) + all-reduce of [4,16,3] partial sums' % (name, world), {'l2': '3.5 GB read per step > L2'})
    line['roofline'] = roofline(8.0 * (B * nz * SHAPE[1] * SHAPE[2] * L), ms / steps, 'cce' if cce else 'dice',
                                '8 B per (voxel,label)', 'cce_vec4u_kernel<4,4>' if cce else 'dice_sums_vec4_kernel')
    line['gpu_launches'] = steps * (2 if cce else 3)
    line['clocks'] = clocks
    del t, p, lab
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cport = cpu_setup()
        rng = np.random.default_rng(0)
        th = np.eye(L, dtype=np.float32)[rng.integers(0, L, (1,) + SHAPE)]
        ph = rng.uniform(0.01, 1, th.shape).astype(np.float32)
        ph /= ph.sum(-1, keepdims=True)
        th, ph = cport.first_touch(th), cport.first_touch(ph)
        fn = (lambda: cport.cce(th, ph)) if cce else (lambda: cport.dice_sums(th, ph))
        line['cpu_baseline'] = cpu_record(fn, V * L, 'elements/s',
                                          'oracle/c %s on ONE [160,192,224,16] volume pair (a quarter of the batch-4 step)'
                                          % ('oracle_cce_f32' if cce else 'oracle_dice_sums_f32'), budget_s=4.0)
    return line


def lc3d_record(args, world, rank, dev, steps, batch=None, cpu=True):
    import numpy as np
    import torch
    from neurite_b200.layers import local_conv3d
    B = batch or args.lc_batch
    I, Cin, Cout = 64, 16, 16
    O = I - 2
    P, F = O ** 3, 27 * Cin
    g = torch.Generator(device=dev).manual_seed(3)
    x = torch.randn((B, I, I, I, Cin), device=dev, generator=g)
    lim = (6.0 / (F + Cout)) ** 0.5
    kernel = (torch.rand((P, F, Cout), device=dev, generator=g) * 2 - 1) * lim
    bias = torch.randn((O, O, O, Cout), device=dev, generator=g)
    sampler = ClockSampler(dev.index).start()
    last = []
    ms = timed_region(lambda: local_conv3d(x, kernel, bias, (3, 3, 3), (1, 1, 1), (O, O, O)), steps, args.warmup, world,
                      last=last)
    clocks = sampler.stop()
    dump_output(args, 'lc3d' if B == 1 else 'lc3d_b%d' % B, last, rank)
    line = base_line('output positions/s, LocallyConnected3D 3^3 16->16 on 64^3, batch %d' % B,
                     P * B * steps / (ms * 1e-3), 'positions/s', world, steps, args.warmup, ms, 'weak',
                     'BASELINE.json configs[3]: LocallyConnected3D 3x3x3, 16->16, input [%d,64,64,64,16], kernel '
                     '[238328,432,16] = 6.59 GB streamed once per step (> L2)' % B)
    line['roofline'] = roofline(4.0 * (P * F * Cout + B * I ** 3 * Cin + B * P * Cout + P * Cout), ms / steps,
                                'lc3d' if B == 1 else ('lc3d_b8' if B == 8 else None), '4*(P*F*Cout + B*in + B*P*Cout + P*Cout)',
                                'lc3d_rows_kernel<4,2>' if B >= 8 else 'lc3d_patch_kernel')
    line['gpu_launches'] = steps
    line['clocks'] = clocks
    del x, kernel, bias
    if rank == 0 and world == 1 and cpu and not args.no_cpu_baseline:
        cport = cpu_setup()
        Is = 26                                              # 24^3 positions: 0.38 GB of weights, streamed once per run
        Os = Is - 2
        rng = np.random.default_rng(0)
        xs = cport.first_touch(rng.standard_normal((1, Is, Is, Is, Cin)).astype(np.float32))
        ks = cport.first_touch((rng.uniform(-1, 1, (Os ** 3, F, Cout)) * lim).astype(np.float32))
        bs = rng.standard_normal((Os, Os, Os, Cout)).astype(np.float32)
        line['cpu_baseline'] = cpu_record(lambda: cport.lc3d(xs, ks, bs, (3, 3, 3)), Os ** 3, 'positions/s',
                                          'oracle/c oracle_lc3d_f32 on a 26^3 input (24^3 = 13824 of the 238328 positions, '
                                          'the same 27.6 KB of private weights per position)', budget_s=4.0)
    return line


def resize_record(args, world, rank, dev, steps):
    import numpy as np
    import torch
    import neurite_b200 as ne
    B = args.batch
    g = torch.Generator(device=dev).manual_seed(5 + rank)
    x = torch.randn((B, 80, 96, 112, 3), device=dev, generator=g)
    lay = ne.layers.Resize(2)
    sampler = ClockSampler(dev.index).start()
    last = []
    ms = timed_region(lambda: lay(x), steps, args.warmup, world, last=last)
    clocks = sampler.stop()
    dump_output(args, 'resize', last, rank)
    line = base_line('output voxels/s, Resize zoom 2 of a half-resolution 3-ch flow to 160x192x224',
                     world * B * V * steps / (ms * 1e-3), 'voxels/s', world, steps, args.warmup, ms, 'weak',
                     'Resize(2) on [%d,80,96,112,3] (reference models.py:803-804)' % B)
    line['roofline'] = roofline(4.0 * 3 * B * V * (1 + 1 / 8), ms / steps, 'resize', '4C/z^3 + 4C per output voxel',
                                'resize3d_kernel')
    line['gpu_launches'] = steps
    line['clocks'] = clocks
    del x
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import interp as ointerp
        cport = cpu_setup()
        xs = np.random.default_rng(0).standard_normal((80, 96, 112, 3)).astype(np.float32)
        # the reference's resize = interpn on an ndgrid of fp32 linspaces (utils.py:237-262)
        lin = [ointerp.tf_linspace_f32(0, s - 1, 2 * s) for s in xs.shape[:3]]
        loc = np.stack(np.meshgrid(*lin, indexing='ij'), -1).astype(np.float32)
        xs, loc = cport.first_touch(xs), cport.first_touch(loc)
        line['cpu_baseline'] = cpu_record(lambda: cport.interpn(xs, loc), V, 'voxels/s',
                                          'oracle/c oracle_interpn_f32 on the explicit linspace grid, ONE [80,96,112,3] -> '
                                          '[160,192,224,3] volume', budget_s=4.0)
    return line


def warp_mc_record(args, world, rank, dev, steps, C=None):
    """Multi-channel warp (the kernel of BASELINE.json configs[4]: a 16-label softmax through the
    SpatialTransformer): z-marching ring kernel, (12 + 8C) B per voxel."""
    import numpy as np
    import torch
    import neurite_b200 as ne
    C = C or args.channels
    B = max(1, min(args.batch, 32 // C))
    g = torch.Generator(device=dev).manual_seed(11 + rank)
    vol = torch.randn((B,) + SHAPE + (C,), device=dev, generator=g)
    flow = torch.rand((B,) + SHAPE + (3,), device=dev, generator=g) * 6 - 3
    if args.flow == 'smooth':
        coarse = torch.randn((B, 3, 10, 12, 14), device=dev, generator=g)
        flow = torch.nn.functional.interpolate(coarse, size=SHAPE, mode='trilinear', align_corners=True)
        flow = (flow / flow.abs().amax() * 3).permute(0, 2, 3, 4, 1).contiguous()
    st = ne.layers.SpatialTransformer(interp_method=args.method)
    sampler = ClockSampler(dev.index).start()
    last = []
    ms = timed_region(lambda: st([vol, flow]), steps, args.warmup, world, last=last)
    clocks = sampler.stop()
    dump_output(args, 'warp_c%d' % C, last, rank)
    line = base_line('voxels/s warped, %d-channel volume (SpatialTransformer %s)' % (C, args.method),
                     world * B * V * steps / (ms * 1e-3), 'voxels/s', world, steps, args.warmup, ms, 'weak',
                     'SpatialTransformer warp of [%d,160,192,224,%d] fp32 (the %d-label softmax of BASELINE.json configs[4]), '
                     'random dense flow %s' % (B, C, C, 'U(-3,3) i.i.d.' if args.flow == 'iid' else 'smooth, max|u|=3'))
    line['roofline'] = roofline((12.0 + 8.0 * C) * B * V, ms / steps, 'warp_c%d' % C,
                                '12 flow + 4C source (each voxel once) + 4C store per voxel', 'warp3d_march_kernel')
    line['gpu_launches'] = steps
    line['clocks'] = clocks
    del vol, flow
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cport = cpu_setup()
        rng = np.random.default_rng(0)
        vs = cport.first_touch(rng.standard_normal((1,) + SHAPE + (C,)).astype(np.float32))
        fs = cport.first_touch(rng.uniform(-3, 3, (1,) + SHAPE + (3,)).astype(np.float32))
        os_ = cport.first_touch(np.zeros(vs.shape, dtype=np.float32))
        line['cpu_baseline'] = cpu_record(lambda: cport.warp(vs, fs, args.method, out=os_), V, 'voxels/s',
                                          'oracle/c oracle_warp_f32, ONE [160,192,224,%d] volume' % C, budget_s=4.0)
    return line


# ---------------------------------------------------------------------------------------
# ONE volume over N ranks: z-slabs + halo exchange (strong scaling, SURVEY.md 8e)
# ---------------------------------------------------------------------------------------
def slab_record(args, world, rank, dev, steps, channels=1, batch=1):
    import torch
    import torch.distributed as dist
    from neurite_b200 import dist as nd, utils
    C, B = channels, batch
    g = torch.Generator(device=dev).manual_seed(77)          # every rank draws the same volume and keeps its planes
    z0, nz = nd.slab_bounds(SHAPE[0], world, rank)
    vol = torch.randn((B,) + SHAPE + (C,), device=dev, generator=g)[:, z0:z0 + nz].contiguous()
    flow = (torch.rand((B,) + SHAPE + (3,), device=dev, generator=g) * 6 - 3)[:, z0:z0 + nz].contiguous()
    halo = 4                                                  # ceil(3) + 1 for U(-3,3): a property of the plan
    model_bytes = (12.0 + 8.0 * C) * B * V
    rec = {'workload': 'ONE batch of %d volume(s) [160,192,224,%d] split in z-slabs over %d rank(s) (%d planes each), flow '
                       'U(-3,3) i.i.d., halo %d planes from each neighbour' % (B, C, world, nz, halo),
           'scaling': 'strong', 'n_gpus': world, 'steps': steps, 'halo_planes': halo,
           'halo_bytes_per_rank_per_step': int(2 * halo * SHAPE[1] * SHAPE[2] * C * 4 * B)}
    name = 'slab' if C == 1 else 'slab_c%d' % C
    if world == 1:
        out = torch.empty_like(vol)
        ms = timed_region(lambda: utils._warp_views(vol, flow, out, SHAPE[0], 0, None, 0, 0), steps, 3, world)
        dump_output(args, name, [out], rank)               # every step overwrites `out`: it holds the last one
        rec['overlap'] = {'ms_per_step': ms / steps, 'value': B * V * steps / (ms * 1e-3), 'unit': 'voxels/s'}
        return rec
    out = torch.empty(tuple(flow.shape[:-1]) + (C,), dtype=torch.float32, device=dev)
    peak, _ = measured_peak()

    def measure(transport):
        plan = nd.SlabWarper(SHAPE[0], halo, transport=transport)
        # the producer of the volume writes its planes straight into the plan's buffer (zero-copy hand-over): the
        # step is exchange + kernels only
        src = plan.source_view(vol)
        src.copy_(vol)
        ms_ov = timed_region(lambda: plan(src, flow, out), steps, 3, world, min_preheat_s=0.1)
        if transport == 'auto':
            dump_output(args, name, [out], rank)           # rank 0's planes of the last step
        plan.check()
        # the two ingredients on their own: the halo exchange (no kernels) and the three launches (no exchange)
        ext, pad = plan._buffers(vol), plan._pad
        mid = ext[:, pad:pad + nz]
        ms_ex = timed_region(lambda: plan._exchange(ext, mid)(), steps, 3, world, min_preheat_s=0.0)

        def kernels_only():
            i_lo, i_hi = plan.lo_pad, nz - plan.hi_pad
            srcx = ext[:, pad - plan.lo_pad:pad + nz + plan.hi_pad]
            plan._kernel(mid, flow[:, i_lo:i_hi], out[:, i_lo:i_hi], z0, z0 + i_lo)
            if i_lo > 0:
                plan._kernel(srcx, flow[:, :i_lo], out[:, :i_lo], z0 - plan.lo_pad, z0)
            if i_hi < nz:
                plan._kernel(srcx, flow[:, i_hi:], out[:, i_hi:], z0 - plan.lo_pad, z0 + i_hi)
        ms_k = timed_region(kernels_only, steps, 3, world, min_preheat_s=0.0)
        plan._err.zero_()
        graph = None
        if plan.active_transport == 'peer':
            # the same step as ONE CUDA-graph replay (no python / launch overhead between its pieces)
            err = None
            try:
                plan.capture(src, flow, out)
            except Exception as ex:                          # noqa: BLE001
                err = '%s: %s' % (type(ex).__name__, str(ex)[:200])
            # the replay contains device-side barriers: every rank must have a graph, or nobody replays
            okf = torch.tensor([0.0 if err else 1.0], device=dev)
            dist.all_reduce(okf, op=dist.ReduceOp.MIN)
            if float(okf.item()) > 0:
                ms_g = timed_region(plan.replay, steps, 3, world, min_preheat_s=0.0)
                plan.check()
                graph = {'ms_per_step': ms_g / steps, 'value': B * V * steps / (ms_g * 1e-3), 'unit': 'voxels/s'}
            else:
                graph = {'error': err or 'capture failed on another rank'}
        return {'transport': plan.active_transport, 'cuda_graph_replay': graph,
                'ms_per_step': ms_ov / steps, 'value': B * V * steps / (ms_ov * 1e-3),
                'unit': 'voxels/s', 'exchange_only_us': ms_ex / steps * 1e3, 'kernels_only_us': ms_k / steps * 1e3,
                'roofline_frac_aggregate': model_bytes / (ms_ov / steps * 1e-3) / 1e9 / (peak * world),
                'limiter': 'the halo exchange' if ms_ex > ms_k else 'the three kernel launches'}
    rec['overlap'] = measure('auto')
    rec['overlap']['what'] = ('SlabWarper: interior planes warped while the halo planes travel; no host sync in the step; '
                              'transport peer = halos pulled out of the neighbours\' symmetric-memory buffers over NVLink, '
                              'nccl = one ncclGroup of send/recv')
    if rec['overlap']['transport'] == 'peer':
        rec['overlap_nccl'] = measure('nccl')
    ser_steps = max(1, steps // 4)
    ms_ser = timed_region(lambda: nd.warp_slab(vol, flow, SHAPE[0], mode='serial', halo=halo), ser_steps, 3, world, min_preheat_s=0.0)
    rec['serial'] = {'steps': ser_steps, 'ms_per_step': ms_ser / ser_steps, 'value': B * V * ser_steps / (ms_ser * 1e-3), 'unit': 'voxels/s',
                     'what': 'round-1 path: NCCL exchange, then one launch, err.item() every step'}
    # strong-scaling reference: the same batch on ONE GPU (no exchange), timed on rank 0's device
    g1 = torch.Generator(device=dev).manual_seed(78)
    vol1 = torch.randn((B,) + SHAPE + (C,), device=dev, generator=g1)
    flow1 = torch.rand((B,) + SHAPE + (3,), device=dev, generator=g1) * 6 - 3
    out1 = torch.empty_like(vol1)
    ms_one = timed_region(lambda: utils._warp_views(vol1, flow1, out1, SHAPE[0], 0, None, 0, 0), ser_steps, 3, world,
                          min_preheat_s=0.0)
    best = rec['overlap']['ms_per_step']
    gr = rec['overlap'].get('cuda_graph_replay') or {}
    if 'ms_per_step' in gr:
        best = min(best, gr['ms_per_step'])
    rec['one_gpu_whole_volume'] = {'ms_per_step': ms_one / ser_steps, 'steps': ser_steps,
                                   'speedup_of_the_slab_plan': (ms_one / ser_steps) / best}
    return rec


def cfg5_record(args, world, rank, dev, steps):
    """BASELINE.json configs[4]: UNet fwd -> SpatialTransformer (16 labels) -> Dice, global batch = N volumes
    (one per GPU), batch-sharded and z-slab-sharded.  The UNet is stock torch/cuDNN (context); the warp and the Dice
    are this repo's kernels and are the part that counts toward the roofline."""
    import torch
    spec = importlib.util.spec_from_file_location('cfg5_example', os.path.join(ROOT, 'examples', 'cfg5_unet_warp_dice.py'))
    ex = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ex)
    group = torch.distributed.group.WORLD if world > 1 else None
    rec = {'workload': 'UNet(16 features, 4 levels, bf16 autocast, cuDNN) fwd -> SpatialTransformer of the 16-label softmax -> '
                       'Dice vs one-hot target, 160x192x224, global batch %d' % max(world, args.cfg5_batch),
           'n_gpus': world, 'steps': steps}
    peak, _ = measured_peak()
    for mode in (('batch', 'slab') if world > 1 else ('batch',)):
        torch.cuda.empty_cache()
        gb = max(world, args.cfg5_batch)                      # global batch
        B = gb if mode == 'slab' else gb // world
        job = ex.Cfg5(mode, B, dev, world, rank, group)
        stage_ms = [0.0, 0.0, 0.0]
        evs = []

        def mark(i):
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            evs.append(e)

        def step_marked():
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            evs.append(e)
            return job.step(mark)
        last = []
        ms = timed_region(lambda: job.step(), steps, 2, world, min_preheat_s=0.0, last=last)
        dump_output(args, 'cfg5_' + mode, last, rank)
        loss = job.step()
        evs.clear()
        for _ in range(3):
            step_marked()
        torch.cuda.synchronize()
        for k in range(0, len(evs), 4):
            for i in range(3):
                stage_ms[i] += evs[k + i].elapsed_time(evs[k + i + 1]) / 3.0
        if job.plan is not None:
            job.plan.check()
        nvox_rank = B * job.nz * SHAPE[1] * SHAPE[2]
        # per-stage times: in slab mode the ranks at the ends of the volume have smaller UNet windows and then WAIT in
        # the halo exchange for their neighbours, so rank 0's 'warp' would mostly be that wait; report the largest
        # UNet time and the SMALLEST warp / Dice times over the ranks (the rank that arrives last does not wait)
        st_t = torch.tensor(stage_ms, dtype=torch.float64, device=dev)
        st_max, st_min = st_t.clone(), st_t.clone()
        if world > 1:
            torch.distributed.all_reduce(st_max, op=torch.distributed.ReduceOp.MAX)
            torch.distributed.all_reduce(st_min, op=torch.distributed.ReduceOp.MIN)
        stage_ms = [float(st_max[0]), float(st_min[1]), float(st_min[2])]
        rec[mode] = {
            'ms_per_step': ms / steps, 'value': gb * steps / (ms * 1e-3), 'unit': 'volumes/s',
            'stage_ms': {'unet_max_over_ranks': stage_ms[0], 'warp_min_over_ranks': stage_ms[1], 'dice_min_over_ranks': stage_ms[2]},
            'transport': job.plan.active_transport if job.plan is not None else None,
            'warp_roofline_frac': 140.0 * nvox_rank / (stage_ms[1] * 1e-3) / 1e9 / peak if stage_ms[1] > 0 else None,
            'dice_roofline_frac': 128.0 * nvox_rank / (stage_ms[2] * 1e-3) / 1e9 / peak if stage_ms[2] > 0 else None,
            'mean_dice_loss': float(loss),
            'parallelism': ('every rank: %d whole volume(s); collective = all-reduce of the scalar loss' % B) if mode == 'batch' else
                           ('every rank: planes [%d,%d) of all %d volumes; UNet on the slab + receptive-field margin (window '
                            '[%d,%d)); %d halo planes of the 16-channel segmentation from each neighbour overlapped with the interior '
                            'warp; all-reduce of the [B,16,3] Dice sums' % (job.z0, job.z0 + job.nz, B, job.w0, job.w1, job.plan.halo if job.plan else 0)),
        }
        del job
    return rec


def bench_mi(args, segs=False):
    """MutualInformation: `mi` = volumes() on B pairs of 160x192x224 volumes (soft quantisation
    fused, 8 B/voxel); `mi_segs` = segs() on two [2,160,192,224,16] probability maps (128 B/voxel)."""
    import torch
    import neurite_b200 as ne
    world, rank, local = dist_setup(args.gpus)
    dev = torch.device('cuda', local)
    m = ne.metrics.MutualInformation(nb_bins=16)
    g = torch.Generator(device=dev).manual_seed(13 + rank)
    if segs:
        B = 2
        x = torch.softmax(torch.randn((B,) + SHAPE + (16,), device=dev, generator=g), -1)
        y = torch.softmax(torch.randn((B,) + SHAPE + (16,), device=dev, generator=g), -1)
        fn, per_voxel, kern = (lambda: m.segs(x, y)), 128.0, 'mi_hist_mma_kernel<1,2,maps,maps>'
    else:
        B = args.batch
        x = torch.rand((B,) + SHAPE + (1,), device=dev, generator=g)
        y = (0.7 * x * x + 0.1 + 0.1 * torch.rand(x.shape, device=dev, generator=g)).clamp_(0, 1)
        fn, per_voxel, kern = (lambda: m.volumes(x, y)), 8.0, 'mi_hist_mma_kernel<1,2,quant,quant>'
    sampler = ClockSampler(local).start()
    last = []
    ms = timed_region(fn, args.steps, args.warmup, world, last=last)
    clocks = sampler.stop()
    dump_output(args, 'mi_segs' if segs else 'mi', last, rank)
    if rank == 0:
        line = base_line('voxels/s, MutualInformation.%s (16 bins), 160x192x224 fp32' % ('segs' if segs else 'volumes'),
                         world * B * V * args.steps / (ms * 1e-3), 'voxels/s', world, args.steps, args.warmup, ms, 'weak',
                         'MutualInformation(nb_bins=16).%s on %d x 160x192x224 (reference metrics.py:41-336); '
                         'min/max + histogram + combine + finalise kernels per step' % ('segs, 16 labels' if segs else 'volumes', B))
        line['dtype'] = 'f32 (3xTF32 tensor-core contraction)'
        line['roofline'] = roofline(per_voxel * B * V, ms / args.steps, 'mi_segs' if segs else 'mi',
                                    '%d B/voxel (two fp32 %s read once; the quantised [V,16] maps never exist)'
                                    % (per_voxel, 'maps' if segs else 'volumes'), kern)
        if not segs:
            line['roofline']['note'] = 'volumes(): bound by issue slots / MUFU (32 exp per voxel pair), not HBM'
        line['gpu_launches'] = args.steps * (4 if segs else 10)
        line['clocks'] = clocks
        if world == 1 and not segs and not args.no_cpu_baseline:
            import numpy as np
            cport = cpu_setup()
            xs = np.random.default_rng(0).uniform(0, 1, (1,) + SHAPE + (1,)).astype(np.float32)
            ys = np.clip(0.7 * xs * xs + 0.1 + 0.1 * np.random.default_rng(1).uniform(0, 1, xs.shape), 0, 1).astype(np.float32)
            xs, ys = cport.first_touch(xs), cport.first_touch(ys)
            line['cpu_baseline'] = cpu_record(
                lambda: cport.mi_channelwise(xs, ys, nb_bins=16), V, 'voxels/s',
                'oracle/c oracle_mi_channelwise_f32 (C99+OpenMP restatement of metrics.py:185-292 with soft_quantize '
                'fused), ONE 160x192x224 volume pair', budget_s=4.0, min_runs=5)
        print(json.dumps(line), flush=True)
    finish(world)


def bench_blur(args):
    """GaussianBlur(sigma=1) (7 taps per axis) of B single-channel 160x192x224 volumes: three separable passes."""
    import torch
    import neurite_b200 as ne
    world, rank, local = dist_setup(args.gpus)
    dev = torch.device('cuda', local)
    B = args.batch
    g = torch.Generator(device=dev).manual_seed(17 + rank)
    x = torch.randn((B,) + SHAPE + (1,), device=dev, generator=g)
    lay = ne.layers.GaussianBlur(sigma=args.sigma)
    sampler = ClockSampler(local).start()
    last = []
    ms = timed_region(lambda: lay(x), args.steps, args.warmup, world, last=last)
    clocks = sampler.stop()
    dump_output(args, 'blur', last, rank)
    if rank == 0:
        line = base_line('voxels/s, GaussianBlur(sigma=%g), 160x192x224 fp32' % args.sigma,
                         world * B * V * args.steps / (ms * 1e-3), 'voxels/s', world, args.steps, args.warmup, ms, 'weak',
                         'GaussianBlur(sigma=%g) on [%d,160,192,224,1] (reference layers.py:251-364): three separable passes'
                         % (args.sigma, B))
        line['roofline'] = roofline(8.0 * B * V, ms / args.steps, 'blur',
                                    '8 B/voxel for the whole blur (read once, write once); the three-pass path moves '
                                    '24 B/voxel, so 0.33 is its ceiling', 'sepconv_col4_kernel x2 + sepconv_row_kernel')
        line['gpu_launches'] = args.steps * 3
        line['clocks'] = clocks
        if world == 1 and not args.no_cpu_baseline:
            import numpy as np
            cport = cpu_setup()
            xs = cport.first_touch(np.random.default_rng(0).standard_normal((1,) + SHAPE + (1,)).astype(np.float32))
            line['cpu_baseline'] = cpu_record(
                lambda: cport.gaussian_blur(xs, args.sigma), V, 'voxels/s',
                'oracle/c oracle_sepconv_axis_f32 x3 (C99+OpenMP restatement of utils.py:665-751), ONE 160x192x224 volume',
                budget_s=4.0, min_runs=5)
        print(json.dumps(line), flush=True)
    finish(world)


def single_op(args, fn):
    import torch
    world, rank, local = dist_setup(args.gpus)
    dev = torch.device('cuda', local)
    rec = fn(args, world, rank, dev, args.steps)
    if rank == 0:
        print(json.dumps(rec), flush=True)
    finish(world)


def finish(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200, help='timed steps of the line\'s own measurement')
    ap.add_argument('--long-steps', type=int, default=200,
                    help='timed steps of the headline\'s long_run and of each sub-record of the default line '
                         '(ops at 1 GPU, slab and slab_c16 at N GPUs)')
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--op', default='warp', choices=['warp', 'dice', 'cce', 'lc3d', 'resize', 'warp_mc', 'warp_slab', 'cfg5',
                                                      'mi', 'mi_segs', 'blur'])
    ap.add_argument('--sigma', type=float, default=1.0)
    ap.add_argument('--batch', type=int, default=8)
    ap.add_argument('--channels', type=int, default=16)
    ap.add_argument('--lc-batch', type=int, default=1)
    ap.add_argument('--slab-batch', type=int, default=1)
    ap.add_argument('--slab-channels', type=int, default=1)
    ap.add_argument('--cfg5-steps', type=int, default=5, help='timed steps of the cfg5 record')
    ap.add_argument('--cfg5-batch', type=int, default=0, help='global batch of --op cfg5 (default: one volume per GPU)')
    ap.add_argument('--method', default='linear', choices=['linear', 'nearest'])
    ap.add_argument('--flow', default='iid', choices=['iid', 'smooth'])
    ap.add_argument('--halo', type=int, default=0)
    ap.add_argument('--e2e-steps', type=int, default=10, help='timed steps of the headline\'s e2e record')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-numpy-baseline', action='store_true')
    ap.add_argument('--no-extras', action='store_true', help='headline only: no ops / slab / cfg5 sub-records')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last timed step of each record computed as '
                         'DIR/<name>.npy (float32; outputs over %d elements as a fixed seeded sample; rank 0\'s '
                         'outputs at N GPUs)' % DUMP_ELEMS)
    args = ap.parse_args()
    if args.impl == 'reference':
        return bench_reference(args)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device -- the product path has no CPU fallback '
                         '(use --impl reference for the CPU port of the reference)')
    if args.op == 'warp':
        return bench_warp(args)
    if args.op in ('mi', 'mi_segs'):
        return bench_mi(args, segs=args.op == 'mi_segs')
    if args.op == 'blur':
        return bench_blur(args)
    single_op(args, {
        'dice': lambda a, w, r, d, k: dice_record(a, w, r, d, k, cce=False),
        'cce': lambda a, w, r, d, k: dice_record(a, w, r, d, k, cce=True),
        'lc3d': lc3d_record, 'resize': resize_record, 'warp_mc': warp_mc_record,
        'warp_slab': lambda a, w, r, d, k: slab_record(a, w, r, d, k, channels=a.slab_channels, batch=a.slab_batch),
        'cfg5': lambda a, w, r, d, k: cfg5_record(a, w, r, d, a.cfg5_steps)}[args.op])


if __name__ == '__main__':
    main()
