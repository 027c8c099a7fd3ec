"""bench.py -- Monte-Carlo free-integration throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    torchrun ... bench.py --gpus N ...          (one rank per GPU, NCCL)

Workload = BASELINE.json configs[1]: free_integration on motion_def-90deg_turn.csv
(true trajectory from the reference's path_gen, frozen in tests/golden/traj_*.npz: n = 1000
samples at 100 Hz), 'mid-accuracy' IMU, ref_frame = 1, 1000 Monte-Carlo runs per GPU
(weak scaling: N GPUs -> 1000 N runs, global run ids rank-independent).

A "step" is one pass of the hot path over that batch: on-device IMU error generation
(Philox) -> strapdown free integration -> per-run end-point errors (K12), then the ensemble
statistics (K3; for N > 1 the fused statistics + peer-memory exchange kernel K3x).  `value` =
runs x samples / device time with inputs resident in HBM; `e2e` = the same through the public
API (Sim.run + error statistics) with HOST buffers, H2D of the trajectory and D2H of the
statistics inside the timed region; `e2e_histories` additionally brings every run's att/pos/vel
history (72 B per run-step) to the host, which is what the reference's Sim.run leaves behind.
L2 is flushed between timed steps.  `extra` carries the other BASELINE configurations measured in
the same process (config 3 sharded over the ranks, config 4 at N = 1) and, for N > 1, the check
that the sharded statistics equal the single-GPU ones.  See DESIGN.md section 7.

--steps K sets the number of steps of every timed loop.  --dump-outputs DIR writes what the last
timed step returned as float64 .npy files: end_err.npy (per-run end-point errors of rank 0's runs,
[1000, 9]) and error_stats.npy (ensemble max|e| / mean / std, [3, 9]).  The inputs are fixed (frozen
trajectory, fixed seed), so two builds can be compared output for output.
"""
import argparse
import ctypes
import glob
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it
_REAL_STDOUT = None


def emit(obj):
    line = (json.dumps(obj) + '\n').encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line)


METRIC = 'MC-runs x timesteps/sec free_integration @100Hz'
UNIT = 'run-steps/s'
RUNS_PER_GPU = 1000
FS = 100.0
SEED = 12345
TRAJ = os.path.join(ROOT, 'tests', 'golden', 'traj_90deg_turn_100hz_rf1.npz')
WORKLOAD = ("free_integration, motion_def-90deg_turn.csv (n=1000 @100Hz), 'mid-accuracy' IMU, "
            "ref_frame=1, 1000 MC runs per GPU")
# what the roofline fields need from an ncu capture of the dominant kernel at THIS workload
# (tools/ncu_summary.py output): FP64 thread-instructions per run-step, DRAM bytes per launch, and the
# launch shape they were counted on -- read at run time, never copied into this file
ROOFLINE_INPUTS = os.path.join(ROOT, 'profiles', 'roofline_inputs_r02.json')
C3_CSV = os.path.join(ROOT, 'tests', 'golden', 'motion_def-long_drive.csv')
C3_RUNS, C3_FS = 100000, 200.0


def common_config(total_runs, n, gpus):
    """The workload, named identically by both arms."""
    return {'workload': WORKLOAD, 'runs': total_runs, 'runs_per_gpu': RUNS_PER_GPU, 'samples': n,
            'global_run_steps': total_runs * n, 'seed': SEED, 'gpus': gpus}


def load_workload():
    g = dict(np.load(TRAJ))
    nav = np.concatenate([g['ref_att'], g['ref_pos'], g['ref_vel']], axis=1)
    return g, np.ascontiguousarray(nav)


def host_info():
    model = ''
    try:
        with open('/proc/cpuinfo') as f:
            for line in f:
                if line.startswith('model name'):
                    model = line.split(':', 1)[1].strip()
                    break
    except OSError:
        pass
    return model, os.cpu_count()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    FIELDS = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
              'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
              'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.FIELDS,
                 '--format=csv,noheader,nounits', '-lms', '50'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line)

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in self.lines:
            f = [x.strip() for x in line.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(nm)
        return {'sm_mhz': statistics.median(sm) if sm else None,
                'sm_max_mhz': max(mx) if mx else None, 'samples': len(sm),
                'reasons': sorted(reasons)}


# ------------------------------------------------------------------ CPU arms ---------------------
def _oracle_c():
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import oracle_c
    return oracle_c


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (its C port,
    oracle/oracle.c -- the NumPy original is timed beside it per core in `cpu_baseline`) on all host
    cores.  A step is the workload repeated `reps` times in ONE call (one thread start per step), sized
    so that a step lasts a few tenths of a second; the value is run-steps per second either way."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    oracle_c = _oracle_c()
    from gnss_ins_sim_b200 import imu_model
    g, nav = load_workload()
    imu = imu_model.IMU(accuracy='mid-accuracy', axis=6, gps=False)
    n = nav.shape[0]
    runs = RUNS_PER_GPU * args.gpus
    ini = g['ini'][None]

    def step(k, reps):
        return oracle_c.mc_free_integration(1, FS, runs * reps, 0, g['ref_gyro'], g['ref_accel'], nav[-1],
                                            imu.gyro_err, imu.accel_err, SEED + k, ini, threads=0)
    step(0, 1)
    t0 = time.perf_counter()
    step(0, 4)
    rate = 4 * runs * n / (time.perf_counter() - t0)
    reps = int(max(1, min(400, round(rate * 0.4 / (runs * n)))))       # ~0.4 s per step
    used = 1
    for k in range(args.warmup):
        _, used = step(k, reps)
    t0 = time.perf_counter()
    for k in range(args.steps):
        err, used = step(args.warmup + k, reps)
    dt = time.perf_counter() - t0
    value = runs * reps * n * args.steps / dt
    model, ncpu = host_info()
    emit({
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt / args.steps * 1e3,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64',
        'data': 'synthetic',
        'config': common_config(runs, n, args.gpus),
        'impl_config': {'workload_repeats_per_step': reps, 'timed_region_s': dt, 'threads': used,
                        'code': 'oracle/oracle.c (C port of the reference path, one run per thread at a time)'},
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': used, 'kind': 'port',
                         'sample': 'the workload (%d runs x %d samples) %d times per step, C port of the '
                                   'reference path, %d threads; host: %s (%s logical cpus)'
                                   % (runs, n, reps, used, model, ncpu)},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    })


def numpy_reference_rate(g, budget_s=6.0):
    """The reference's own NumPy path on ONE host core of this box, if the unmodified package
    travelled with the tree (baseline/_ref, a pip --target install made in the build container;
    git-ignored): Sim.run(R) of demo_free_integration's configuration, noise generation + per-step
    Python loop, no plots.  Returns a dict or None."""
    ref = os.path.join(ROOT, 'baseline', '_ref')
    if not os.path.isdir(os.path.join(ref, 'gnss_ins_sim')):
        return None
    code = r'''
import sys, time, json, io, contextlib
sys.path.insert(0, %r)
import numpy as np
from gnss_ins_sim.sim import imu_model, ins_sim
from demo_algorithms import free_integration
g = dict(np.load(%r))
md = %r
imu = imu_model.IMU(accuracy='mid-accuracy', axis=6, gps=False)
ini = g['ini']
def go(R):
    algo = free_integration.FreeIntegration(ini)
    sim = ins_sim.Sim([%f, 0.0, 0.0], md, ref_frame=1, imu=imu, mode=None, env=None, algorithm=algo)
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):
        sim.run(R)
    return time.perf_counter() - t0, sim.dmgr.get_data(['pos'])[0]['algo0_0'].shape[0]
go(1)
t, n = go(4)
R = int(max(4, min(512, %f / (t / 4))))
t, n = go(R)
print(json.dumps({'runs': R, 'samples': n, 'seconds': t, 'run_steps_per_s': R * n / t}))
''' % (ref, TRAJ, os.path.join(ROOT, 'tests', 'golden', 'motion_def-90deg_turn.csv'), FS, budget_s)
    try:
        out = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, timeout=120)
        d = json.loads(out.stdout.strip().splitlines()[-1])
        # path_gen (about 10 s of pure Python for this trajectory) is outside Sim.run's Monte-Carlo loop
        # but inside Sim.run: report what Sim.run costs per run beyond it by timing two sizes
        return d
    except Exception as e:      # the reference is optional on the box
        sys.stderr.write('numpy reference not timed: %s\n' % e)
        return None


def cpu_baseline_sample(g, nav, imu, budget_s=4.0):
    """Rank 0, N = 1: the C port timed on the host cores on a bounded sample of the workload, and
    the NumPy reference itself on one core."""
    oracle_c = _oracle_c()
    n = nav.shape[0]
    ini = g['ini'][None]

    def go(runs, threads):
        t0 = time.perf_counter()
        _, used = oracle_c.mc_free_integration(1, FS, runs, 0, g['ref_gyro'], g['ref_accel'],
                                               nav[-1], imu.gyro_err, imu.accel_err, SEED, ini,
                                               threads=threads)
        return time.perf_counter() - t0, used
    go(64, 0)
    t_probe, used = go(512, 0)
    rate = 512 * n / t_probe
    runs = int(max(512, min(2_000_000, rate * budget_s / n)))
    t, used = go(runs, 0)
    t1, _ = go(256, 1)
    model, ncpu = host_info()
    value, per_core = runs * n / t, 256 * n / t1
    out = {'value': value, 'unit': UNIT, 'cores': used, 'kind': 'port',
           'per_core_value': per_core, 'effective_cores': round(value / per_core, 1),
           # the GPU box's host is shared between the boxes of the pod: the threads rarely get a core each
           'sample': '%d runs x %d samples of the same workload (%.1f s), C port of the reference '
                     'path (oracle/oracle.c), %d threads; host: %s (%s logical cpus)'
                     % (runs, n, t, used, model, ncpu)}
    ref = numpy_reference_rate(g)
    if ref is not None:
        out['numpy_reference'] = {
            'value': ref['run_steps_per_s'], 'unit': UNIT, 'cores': 1, 'kind': 'reference',
            'sample': 'the unmodified reference (baseline/_ref): ins_sim.Sim.run(%d) with its '
                      'FreeIntegration plugin on this workload (%d samples), %.1f s on one core of this host, '
                      'path_gen included as Sim.run includes it' % (ref['runs'], ref['samples'], ref['seconds'])}
    else:
        out['numpy_reference'] = {'unavailable': 'baseline/_ref (pip --target install of the reference) '
                                                 'is not in this tree'}
    return out


# ------------------------------------------------------------------ B200 arm ---------------------
def dump_outputs(path, arrays):
    """--dump-outputs: one float64 .npy per array the timed step returned."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + '.npy'), np.ascontiguousarray(a, dtype=np.float64))


def roofline_inputs(lanes, shape):
    """FP64 instructions per run-step and DRAM bytes per launch of the dominant kernel, from the
    committed ncu summary named in profiles/roofline_inputs_r02.json -- valid only for the launch
    shape they were counted on."""
    try:
        with open(ROOFLINE_INPUTS) as f:
            d = json.load(f)
    except (OSError, ValueError):
        return None, 'profiles/roofline_inputs_r02.json missing'
    if int(d.get('lanes_per_run', -1)) != int(lanes) or d.get('shape') != shape:
        return None, 'capture is for lanes=%s shape=%s, this run used lanes=%s shape=%s' % (
            d.get('lanes_per_run'), d.get('shape'), lanes, shape)
    return d, d.get('source')


def run_b200(args):
    import torch
    import torch.distributed as td
    from gnss_ins_sim_b200 import engine, imu_model, dist, _lib, build as b2build, pathgen
    from gnss_ins_sim_b200.sim import Sim
    from gnss_ins_sim_b200.free_integration import FreeIntegration

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (no CPU fallback)')
    torch.cuda.set_device(local)
    if world > 1:
        td.init_process_group('nccl', device_id=torch.device('cuda', local))
    assert world == args.gpus, 'launch with torchrun --nproc-per-node %d' % args.gpus

    lib = _lib.load()
    g, nav_h = load_workload()
    imu = imu_model.IMU(accuracy='mid-accuracy', axis=6, gps=False)
    n = nav_h.shape[0]
    R = RUNS_PER_GPU
    total_runs = R * world
    ref_gyro, ref_accel = engine.to_device(g['ref_gyro']), engine.to_device(g['ref_accel'])
    nav, ini = engine.to_device(nav_h), engine.to_device(g['ini'][None])
    cfg = engine.make_mc_config(1, FS, n, R, SEED, imu.gyro_err, imu.accel_err, 1, 9,
                                run_offset=rank * R, ini_offset=rank * R, lanes_per_run=args.lanes)
    res = engine.McResult()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')   # > 126 MB L2
    sms = torch.cuda.get_device_properties(local).multi_processor_count
    lanes_used = args.lanes or lib.b2ins_diag_auto_lanes(R, 1, sms)
    shape_used = _lib.mc_shape(lanes_used, 1)

    merger = p2p = None
    exchange = 'none'
    if world > 1:
        try:        # K3x: statistics + exchange + merge fused in one kernel over NVLink peer memory
            p2p = dist.P2PStats(9)
            exchange = 'fused peer-memory kernel (K3x)'
        except Exception as e:     # no symmetric memory on this box: NCCL all_gather of 28 doubles
            sys.stderr.write('P2PStats unavailable (%s); using NCCL all_gather\n' % e)
            merger = dist.StatsMerger(9)
            exchange = 'NCCL all_gather + host merge'

    def step():
        engine.mc_free_integration(cfg, ref_gyro, ref_accel, nav, ini, out=res)
        if world == 1:
            return engine.error_stats(res.end_err)
        if p2p is not None:
            return p2p(res.end_err, R)          # stays on the device, like the N = 1 step: no host sync per step
        return merger(engine.error_stats(res.end_err), R)

    def barrier():
        if world > 1:
            td.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device='cuda')
        if world > 1:
            td.all_reduce(t, op=td.ReduceOp.MAX)
        return float(t.item())

    for _ in range(max(args.warmup, 3)):
        stats = step()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    evs = []
    barrier()
    for _ in range(args.steps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        stats = step()
        e1.record()
        evs.append((e0, e1))
    barrier()
    clocks = sampler.stop()
    dev_ms = allmax(sum(a.elapsed_time(b) for a, b in evs))
    value = total_runs * n * args.steps / (dev_ms * 1e-3)
    stats = stats.cpu().numpy().copy() if hasattr(stats, 'cpu') else stats
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {'end_err': res.end_err.cpu().numpy(), 'error_stats': stats})
    k3x_timed_out = bool(p2p.timed_out()) if p2p is not None else False

    # ---- N > 1: the sharded statistics against ONE GPU doing all the runs -------------------
    parity = None
    if world > 1:
        parity = {'workload': 'config 2, %d runs' % total_runs, 'k3x_timed_out': k3x_timed_out}
        if rank == 0:
            cfg_all = engine.make_mc_config(1, FS, n, total_runs, SEED, imu.gyro_err, imu.accel_err, 1, 9,
                                            lanes_per_run=args.lanes)
            one = engine.mc_free_integration(cfg_all, ref_gyro, ref_accel, nav, ini)
            st1 = engine.error_stats(one.end_err).cpu().numpy()
            parity['max_rel_diff'] = float(np.max(np.abs(stats - st1) / np.maximum(np.abs(st1), 1e-300)))

    # ---- dominant kernel alone: launch duration -> roofline --------------------------------
    kev = []
    for _ in range(args.steps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        engine.mc_free_integration(cfg, ref_gyro, ref_accel, nav, ini, out=res)
        e1.record()
        kev.append((e0, e1))
    torch.cuda.synchronize()
    k_ms = statistics.mean(a.elapsed_time(b) for a, b in kev)
    # algorithmic HBM bytes of one launch: the shared trajectory once (n x 48 B), the last
    # ref_nav row, the initial state, and 72 B of end-point error per run (DESIGN.md 6)
    alg_bytes = n * 48 + 72 + 72 + R * 72
    peaks = {}
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            peaks = json.load(f)
    except OSError:
        pass
    hbm_peak = float(peaks.get('hbm_gbs', 6650.0))
    achieved = alg_bytes / (k_ms * 1e-3) / 1e9
    dfma = ctypes.c_double(0.0)
    _lib.check(lib.b2ins_diag_dfma_rate(ctypes.byref(dfma)))
    k_rate = R * n / (k_ms * 1e-3)
    rin, rsrc = roofline_inputs(lanes_used, shape_used)
    fp64 = {'bound': 'fp64-issue', 'peak_dfma_per_s': dfma.value, 'peak_source': 'measured live '
            '(b2ins_diag_dfma_rate)', 'kernel_run_steps_per_s': k_rate,
            'dfma_slots_per_run_step': dfma.value / k_rate, 'lanes_per_run': lanes_used,
            'launch_shape': shape_used, 'inputs_from': rsrc}
    traffic = None
    if rin is not None:
        fp64['fp64_inst_per_run_step'] = rin['fp64_thread_instructions_per_run_step']
        fp64['frac'] = rin['fp64_thread_instructions_per_run_step'] * k_rate / dfma.value
        fp64['frac_note'] = ('FP64 thread-instructions issued / measured FP64-FMA issue rate.  1000 runs '
                             'put ONE attitude warp on an SM: the serial recurrence is bound by the '
                             'dependent-issue latency of that warp (8.8 cycles per dependent DFMA, '
                             'profiles/ilp_probe_r02.jsonl), not by the pipe')
        if 'fp64_thread_instructions_per_run_step_one_lane' in rin:
            # the same count for ONE lane per run: the share of the issued FP64 work that is not a
            # replica of another lane's (lane groups replicate the strapdown step)
            fp64['fp64_inst_per_run_step_one_lane'] = rin['fp64_thread_instructions_per_run_step_one_lane']
            fp64['frac_nonreplicated'] = (rin['fp64_thread_instructions_per_run_step_one_lane'] * k_rate
                                          / dfma.value)
        traffic = rin.get('dram_bytes_per_launch')
    else:
        fp64['frac'] = None

    if args.quick:
        if rank == 0:
            emit({'metric': METRIC, 'value': value, 'unit': UNIT, 'quick': True,
                  'ms_per_step': dev_ms / args.steps, 'kernel_ms': k_ms, 'lanes_per_run': lanes_used,
                  'launch_shape': shape_used})
        return
    # ---- e2e: public API, host buffers, copies inside the timed region -----------------
    # the step's inputs live in PINNED host memory (numpy views of pinned tensors)
    pinned = {k: torch.from_numpy(np.ascontiguousarray(g[k])).pin_memory()
              for k in ('time', 'ref_pos', 'ref_vel', 'ref_att', 'ref_accel', 'ref_gyro')}
    traj_host = {k: v.numpy() for k, v in pinned.items()}

    def e2e_step(histories=False):
        algo = FreeIntegration(g['ini'], lanes_per_run=args.lanes)
        sim = Sim([FS, 0.0, 0.0], traj_host, ref_frame=1, imu=imu, algorithm=algo, seed=SEED,
                  lanes_per_run=args.lanes)
        sim.run(total_runs)
        st = sim.get_error_stats('pos', err_stats_start=-1)
        if histories:
            return st, sim.histories()
        return st

    def timed_e2e(histories, steps):
        for _ in range(3):
            e2e_step(histories)
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            e2e_step(histories)
        barrier()
        return total_runs * n * steps / allmax(time.perf_counter() - t0)

    e2e_value = timed_e2e(False, args.steps)
    e2e_hist_value = timed_e2e(True, args.steps)
    # plan path (N = 1): true IMU samples + last ref_nav row + initial state up,
    # statistics + per-run end-point errors down
    h2d = (n * 6 + 9 + 9) * 8
    d2h = (27 + R * 9) * 8

    # ---- the other BASELINE configurations, in the same process ----------------------------
    extra = {'multi_gpu_parity': parity} if parity is not None else {}
    extra['config3'] = config3_block(world, rank, args, dfma.value)
    if world == 1 and not args.no_config4:
        extra['config4'] = config4_block()
    extra['config5'] = config5_block(world, rank, args)
    if world > 1 and rank == 0:
        bad = [k for k, v in (('config2', parity), ('config3', extra['config3'].get('multi_gpu_parity')))
               if v and (v.get('k3x_timed_out') or v.get('max_rel_diff', 0.0) > 1e-9)]
        if bad:
            raise SystemExit('sharded statistics differ from the single-GPU ones: %s %s' % (bad, extra))

    out = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
        'warmup': max(args.warmup, 3), 'ms_per_step': dev_ms / args.steps,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64',
        'data': 'synthetic',
        'config': common_config(total_runs, n, world),
        'impl_config': {'l2_flush_between_steps': True, 'lanes_per_run': lanes_used,
                        'lanes_source': 'forced (--lanes)' if args.lanes else 'b2ins_diag_auto_lanes',
                        'launch_shape': shape_used,
                        'parallelism': 'runs sharded x%d; statistics exchange: %s' % (world, exchange),
                        'library': b2build.lib_info()},
        'clocks': clocks,
        'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': h2d,
                'd2h_bytes_per_step': d2h, 'api': 'gnss_ins_sim_b200.sim.Sim.run + get_error_stats'},
        'e2e_histories': {'value': e2e_hist_value, 'unit': UNIT, 'h2d_bytes_per_step': h2d + n * 15 * 8,
                          'd2h_bytes_per_step': d2h + R * n * 72,
                          'api': 'Sim.run + get_error_stats + Sim.histories(): att/pos/vel of every run '
                                 '([R, n, 3] x 3, what the reference Sim.run leaves in its data manager)'},
        # per step: the K12 kernel + stats_small_kernel (N = 1) / stats_exchange_kernel (N > 1)
        'gpu_launches': args.steps * 2,
        'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': hbm_peak, 'unit': 'GB/s',
                     'frac': achieved / hbm_peak, 'traffic': traffic,
                     'peak_source': 'MEASURED_PEAKS.json' if peaks else 'fallback',
                     'kernel': 'mc_av_kernel (K12, attitude / velocity split form)' if shape_used == '6,2,0' else 'mc_spec_kernel (K12)', 'kernel_ms': k_ms,
                     'algorithmic_bytes_per_launch': alg_bytes,
                     'note': 'K12 reads the shared trajectory once and writes 72 B per run: it is bound '
                             'by FP64 issue / dependent-issue latency, not by HBM; see roofline_fp64'},
        'roofline_fp64': fp64,
        'accuracy': {'end_point_rmse': {
            'att_rad': np.sqrt(stats[1, 0:3] ** 2 + stats[2, 0:3] ** 2).tolist(),
            'pos_m': np.sqrt(stats[1, 3:6] ** 2 + stats[2, 3:6] ** 2).tolist(),
            'vel_mps': np.sqrt(stats[1, 6:9] ** 2 + stats[2, 6:9] ** 2).tolist()},
            'parity': 'tests/test_gpu_parity.py: <= 1e-6 rel vs the reference on identical draws'},
        'extra': extra,
    }
    if rank == 0 and world == 1:
        out['cpu_baseline'] = cpu_baseline_sample(g, nav_h, imu)
    if rank == 0:
        emit(out)
    if world > 1:
        td.destroy_process_group()


def config3_block(world, rank, args, dfma_rate):
    """BASELINE config 3: motion_def-long_drive.csv @200 Hz (n = 193 036), 'low-accuracy' IMU,
    ref_frame 0, 100 000 runs sharded over the ranks (strong scaling: this rank's share is
    100 000 / N runs).  Trajectory: host path generator on rank 0, broadcast once.  Timed: the fused
    kernel + statistics on the device (max over ranks), and the wall time including path generation
    and the broadcast.  Under N > 1 rank 0 also does all 100 000 runs alone and the merged statistics
    must agree."""
    import torch
    import torch.distributed as td
    from gnss_ins_sim_b200 import engine, imu_model, dist, pathgen
    from gnss_ins_sim_b200.sim import trajectory_from_motion_def
    runs_total = args.c3_runs
    t_wall0 = time.perf_counter()
    traj, t_path = None, 0.0
    if rank == 0:
        t0 = time.perf_counter()
        traj = trajectory_from_motion_def(C3_FS, C3_CSV, 0)
        t_path = time.perf_counter() - t0
    t0 = time.perf_counter()
    traj = dist.broadcast_trajectory(traj)
    t_bcast = time.perf_counter() - t0
    n = traj['ref_gyro'].shape[0]
    ini = pathgen.parse_motion(C3_CSV)[0]
    imu = imu_model.IMU(accuracy='low-accuracy', axis=6, gps=False)
    nav_h = np.ascontiguousarray(np.concatenate([traj['ref_att'], traj['ref_pos'], traj['ref_vel']], axis=1))
    dev = [engine.to_device(a) for a in (traj['ref_gyro'], traj['ref_accel'], nav_h, ini[None])]
    lo, hi = dist.shard(runs_total, rank, world)
    seed = 3

    def launch(r0, r1):
        cfg = engine.make_mc_config(0, C3_FS, n, r1 - r0, seed, imu.gyro_err, imu.accel_err, 1, 9,
                                    run_offset=r0, ini_offset=r0, lanes_per_run=args.lanes)
        res = engine.mc_free_integration(cfg, *dev)
        return res, engine.error_stats(res.end_err)
    # warm-up on a short prefix of the trajectory would be another kernel shape only in n: 64 runs
    launch(lo, min(hi, lo + 64))
    torch.cuda.synchronize()
    if world > 1:
        td.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    res, st_local = launch(lo, hi)
    e1.record()
    torch.cuda.synchronize()
    ms_local = e0.elapsed_time(e1)
    t = torch.tensor([ms_local], dtype=torch.float64, device='cuda')
    if world > 1:
        td.all_reduce(t, op=td.ReduceOp.MAX)
    ms = float(t.item())
    merged = dist.combine_local_stats(st_local.cpu().numpy(), hi - lo)
    wall = time.perf_counter() - t_wall0
    rate = runs_total * n / (ms * 1e-3)
    out = {'workload': "free_integration, motion_def-long_drive.csv (n=%d @200Hz), 'low-accuracy' IMU, "
                       "ref_frame=0, %d MC runs sharded over %d GPU(s)" % (n, runs_total, world),
           'runs': runs_total, 'runs_this_rank': hi - lo, 'samples': n, 'scaling': 'strong',
           'device_ms_max_over_ranks': ms, 'run_steps_per_s': rate,
           'path_gen_s': t_path, 'broadcast_s': t_bcast, 'wall_s_incl_path_gen_broadcast_upload': wall,
           'pos_std_rad_rad_m': merged[2, 3:6].tolist(),
           'fp64_issue_rate_dfma_per_s': dfma_rate}
    if world > 1:
        par = {'workload': 'config 3, %d runs' % runs_total}
        if rank == 0:
            _, st1 = launch(0, runs_total)
            st1 = st1.cpu().numpy()
            par['max_rel_diff'] = float(np.max(np.abs(merged - st1) / np.maximum(np.abs(st1), 1e-300)))
        out['multi_gpu_parity'] = par
    return out


def config4_block():
    """BASELINE config 4 (N = 1): static 10 h @400 Hz (n = 14.4 M), 'low-accuracy' IMU, 256 runs,
    Allan deviation of the 6 channels through Sim.run (noise generation + tau-binning on the device)."""
    import torch
    from gnss_ins_sim_b200 import imu_model
    from gnss_ins_sim_b200.sim import Sim
    from gnss_ins_sim_b200.allan_analysis import Allan
    runs, n, fs = 256, 14400000, 400.0
    # motion_def-static.csv stretched to 10 h: a type-1 zero command gives constant true IMU samples
    # (pathgen.py:198-200, 331-411): specific force of the tilted rest pose, zero rates
    ref_accel = np.tile(np.array([4.9, 0.0, -8.487]), (n, 1))
    z = np.zeros((n, 3))
    traj = {'ref_pos': z, 'ref_vel': z, 'ref_att': z, 'ref_accel': ref_accel, 'ref_gyro': z}
    imu = imu_model.IMU(accuracy='low-accuracy', axis=6, gps=False)
    sim = Sim([fs, 0.0, 0.0], traj, ref_frame=1, imu=imu, algorithm=Allan(), seed=1)
    sim.run(2)
    torch.cuda.synchronize()
    times = []
    for _ in range(2):      # the first pass also pays for the device allocations of the run blocks
        t0 = time.perf_counter()
        sim.run(runs)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    ad = sim.get_data(['ad_gyro'])[0]['algo0_0']
    return {'workload': "Allan variance: static 10 h @400Hz (n=14.4M), 'low-accuracy' IMU, 256 runs x 6 channels",
            'runs': runs, 'samples': n, 'channels': 6, 'ntau': int(ad.shape[0]),
            'seconds': times[-1], 'seconds_first_pass': times[0],
            'sample_channels_per_s': runs * n * 6 / times[-1],
            'api': 'Sim.run(256) with the Allan plugin (device noise generation + tau-binning)'}


def config5_block(world, rank, args):
    """BASELINE config 5: loosely-coupled 15-state GNSS/INS filter, motion_def-ins.csv @100 Hz with GPS at
    10 Hz (n = 73 250, 7 325 GPS samples), demo_ins_loose.py's IMU, 10 000 runs sharded over the ranks.
    The reference algorithm is a stub, so parity is unpinned: the record carries the filter's consistency
    (NEES, 3-sigma containment) beside the time."""
    import torch
    import torch.distributed as td
    from gnss_ins_sim_b200 import imu_model, dist
    from gnss_ins_sim_b200.sim import Sim
    from gnss_ins_sim_b200.ins_loose import InsLoose
    runs_total = args.c5_runs
    acc = {'gyro_b': np.zeros(3), 'gyro_arw': np.array([0.25, 0.25, 0.25]),
           'gyro_b_stability': np.array([3.5, 3.5, 3.5]), 'gyro_b_corr': np.array([100.0, 100.0, 100.0]),
           'accel_b': np.zeros(3), 'accel_vrw': np.array([0.03119, 0.03009, 0.04779]),
           'accel_b_stability': np.array([4.29e-5, 5.72e-5, 8.02e-5]),
           'accel_b_corr': np.array([200.0, 200.0, 200.0])}               # demo_ins_loose.py:28-37
    imu = imu_model.IMU(accuracy=acc, axis=6, gps=True)
    csv = os.path.join(ROOT, 'tests', 'golden', 'motion_def-ins.csv')
    t0 = time.perf_counter()
    sim = Sim([100.0, 10.0, 0.0], csv, ref_frame=0, imu=imu, algorithm=InsLoose(), seed=5)
    sim.run(min(64 * world, runs_total))                 # trajectory, uploads, kernel load
    torch.cuda.synchronize()
    t_setup = time.perf_counter() - t0
    if world > 1:
        td.barrier()
    t0 = time.perf_counter()
    sim.run(runs_total)
    torch.cuda.synchronize()
    dt_local = time.perf_counter() - t0
    t = torch.tensor([dt_local], dtype=torch.float64, device='cuda')
    if world > 1:
        td.all_reduce(t, op=td.ReduceOp.MAX)
    dt = float(t.item())
    n = sim.data['time'].shape[0]
    c = sim.ekf_consistency()
    st = sim.get_error_stats('pos', -1, extra_opt='ned')
    return {'workload': 'ins_loose 15-state loosely-coupled GNSS/INS EKF, motion_def-ins.csv (n=%d @100Hz, GPS '
                        '@10Hz), %d MC runs sharded over %d GPU(s)' % (n, runs_total, world),
            'runs': runs_total, 'samples': n, 'seconds_max_over_ranks': dt, 'run_steps_per_s': runs_total * n / dt,
            'setup_s_path_gen_upload_warmup': t_setup,
            'parity': 'unpinned: the reference algorithm is a stub (ins_loose.py:124-134); kernel == spec in '
                      'tests/test_ekf.py',
            'consistency_this_rank': {'nees_pos_vel_att_mean': c['nees'].mean(0).tolist(),
                                      'inside_3sigma_min_over_states': float(c['inside3'].mean(0).min()),
                                      'gps_epochs': c['epochs']},
            'end_point_pos_ned_std_m': np.asarray(st['std']).tolist(),
            'api': 'Sim.run(%d) with the InsLoose plugin' % runs_total}


def main():
    # Libraries (NCCL's version banner, torchrun notices) write to fd 1; the contract is ONE JSON
    # line on stdout, so everything else is sent to stderr and the line is written to the saved fd.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--lanes', type=int, default=0, help='lanes per run (0 = auto)')
    ap.add_argument('--quick', action='store_true',
                    help='device-timed part only (for runs under a profiler): no e2e, no cpu baseline')
    ap.add_argument('--c3-runs', type=int, default=C3_RUNS, help='Monte-Carlo runs of the config-3 block')
    ap.add_argument('--no-config4', action='store_true')
    ap.add_argument('--c5-runs', type=int, default=10000, help='Monte-Carlo runs of the config-5 block')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the last timed step\'s end-point errors and statistics to DIR/*.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
