"""CPU-side tests (no GPU): the C ABI is complete, the C oracle is pinned to the
reference's golden vectors, the host mirror of the reference interface behaves like the
reference, the product fails loudly without a CUDA device, and the N > 1 host logic works
over gloo with world_size 2."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import oracle_np as onp
import oracle_c
from conftest import ROOT, allan_golden, load_golden, assert_close

TIGHT = 1e-12


# ------------------------------------------------------------------ C ABI ------
def _declared_functions():
    text = open(os.path.join(ROOT, 'include', 'b2ins.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(b2ins_[a-z0-9_]+)\s*\(', text)))


def test_abi_exports_every_declared_symbol():
    from gnss_ins_sim_b200 import _lib
    lib = _lib.load()
    names = _declared_functions()
    assert len(names) >= 18
    raw = ctypes.CDLL(_lib.lib_path())
    for nm in names:
        assert hasattr(raw, nm), 'libb2ins.so does not export %s' % nm
        assert nm in _lib.SIGNATURES, 'python binding misses %s' % nm
    assert sorted(_lib.SIGNATURES) == names
    assert lib.b2ins_version() == 100


def test_abi_structs_match_header_layout():
    from gnss_ins_sim_b200 import _lib
    assert ctypes.sizeof(_lib.SensorErr) == 96
    assert ctypes.sizeof(_lib.Vib) == 48
    assert ctypes.sizeof(_lib.McConfig) == 416        # + dump_quat
    assert _lib.McConfig.dump_stride.offset == 372 and _lib.McConfig.dump_quat.offset == 408
    assert _lib.McConfig.dump_runs.offset == 360 and _lib.McConfig.algo.offset == 368
    assert _lib.McConfig.ref_odo.offset == 392


def test_allan_num_tau_matches_reference_rule():
    from gnss_ins_sim_b200 import engine
    for n, fs in ((180000, 100.0), (7351, 50.0), (800, 100.0), (14400000, 400.0), (9, 1.0),
                  (899, 100.0), (900, 100.0), (1000, 100.0), (123457, 200.0)):
        assert engine.allan_num_tau(n, fs) == onp.allan_multipliers(n, fs), (n, fs)
    assert len(engine.allan_num_tau(14400000, 400.0)) == 55


def test_product_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        # the checks need a process that sees no device: run this test again in one with the GPU hidden
        r = subprocess.run([sys.executable, '-m', 'pytest', '-q', '-p', 'no:cacheprovider',
                            '%s::test_product_fails_loudly_without_gpu' % os.path.abspath(__file__)],
                           cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=''),
                           capture_output=True, text=True)
        assert r.returncode == 0 and '1 passed' in r.stdout, r.stdout + r.stderr
        return
    from gnss_ins_sim_b200 import engine, _lib
    from gnss_ins_sim_b200.free_integration import FreeIntegration
    algo = FreeIntegration(np.zeros(9))
    with pytest.raises((_lib.B2insError, RuntimeError, AssertionError)):
        algo.run([1, 100.0, np.zeros((10, 3)), np.zeros((10, 3))])
    with pytest.raises(_lib.B2insError):
        engine.error_stats(torch.zeros(4, 9, dtype=torch.float64))
    # the host entry points report the CUDA failure instead of computing on the CPU
    lib = _lib.load()
    x = np.zeros((1, 10, 3))
    ini = np.zeros((1, 9))
    rc = lib.b2ins_free_integration_f64_host(1, 100.0, 1, 10, _lib.host_ptr(x), _lib.host_ptr(x), 0,
                                             _lib.host_ptr(ini), 1, 9, 0, 1, _lib.host_ptr(x.copy()),
                                             _lib.host_ptr(x.copy()), _lib.host_ptr(x.copy()), 0)
    assert rc == _lib.ERR_CUDA and b'' != lib.b2ins_last_error()


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, 'gnss_ins_sim_b200')
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith('.py'):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r'^\s*(import|from)\s+oracle', text, flags=re.M), f
                for token in ('oracle_np', 'oracle_c', 'liboracle', 'oracle/'):
                    assert token not in text, (f, token)
            if f.endswith(('.cu', '.cuh')):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r'#include\s+"[^"]*oracle', text), f


# ------------------------------------------------------------------ C oracle ----
@pytest.mark.parametrize('name', ['bosch', 'nxp'])
def test_c_oracle_logged_data(name):
    g = load_golden('logged_%s.npz' % name)
    att, pos, vel = oracle_c.free_integration(0, float(g['fs']), g['gyro'][None], g['accel'][None],
                                              g['ini'][None], earth_rot=False)
    assert_close(att[0], g['att'], TIGHT, what='att')
    assert_close(pos[0], g['pos'], TIGHT, what='pos')
    assert_close(vel[0], g['vel'], TIGHT, what='vel')


def _errs(g):
    return ({'b': g['gyro_b'], 'b_drift': g['gyro_b_drift'], 'b_corr': g['gyro_b_corr'],
             'arw': g['gyro_arw']},
            {'b': g['accel_b'], 'b_drift': g['accel_b_drift'], 'b_corr': g['accel_b_corr'],
             'vrw': g['accel_vrw']})


@pytest.mark.parametrize('tag', ['90deg_mid_rf1', '90deg_mid_rf0', '90deg_low_rf1_run1000'])
def test_c_oracle_philox_stream_through_reference(tag):
    g = load_golden('philox_%s.npz' % tag)
    ge, ae = _errs(g)
    fs, rf = float(g['fs']), int(g['ref_frame'])
    gyro, accel = oracle_c.imu_noise(fs, g['ref_gyro'], g['ref_accel'], ge, ae, int(g['seed']),
                                     g['run_ids'])
    assert_close(gyro, g['gyro'], TIGHT, what='gyro')
    assert_close(accel, g['accel'], TIGHT, what='accel')
    R = gyro.shape[0]
    att, pos, vel = oracle_c.free_integration(rf, fs, gyro, accel, np.tile(g['ini'], (R, 1)))
    assert_close(att, g['att'], 1e-10, what='att')
    assert_close(pos, g['pos'], 1e-10, what='pos')
    assert_close(vel, g['vel'], 1e-10, what='vel')
    nav_end = np.concatenate([g['ref_att'][-1], g['ref_pos'][-1], g['ref_vel'][-1]])
    err, used = oracle_c.mc_free_integration(rf, fs, R, int(g['run_ids'][0]), g['ref_gyro'],
                                             g['ref_accel'], nav_end, ge, ae, int(g['seed']),
                                             g['ini'][None], threads=2)
    st = oracle_c.array_stats(err)
    for k, key in enumerate(('max', 'avg', 'std')):
        gs = np.concatenate([g['stat_att_euler_' + key], g['stat_pos_' + key], g['stat_vel_' + key]])
        assert_close(st[k], gs, 1e-7, 1e-3, what=key)


def test_c_oracle_allan_and_philox_kat():
    g = allan_golden()
    avar, tau = oracle_c.allan_var(g['x'], float(g['fs']))
    assert_close(avar, g['avar'], 1e-10, 0.0, 'avar')
    assert_close(tau, g['tau'], 1e-15, 0.0, 'tau')
    c = (ctypes.c_uint32 * 4)(0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344)
    oracle_c.load().orc_philox(c, ctypes.c_uint32(0xa4093822), ctypes.c_uint32(0x299f31d0))
    assert list(c) == [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


# ------------------------------------------------------------------ imu_model ---
def test_imu_profiles_equal_the_reference_values():
    from gnss_ins_sim_b200 import imu_model
    for tag, grade in (('90deg_mid_rf1', 'mid-accuracy'), ('90deg_low_rf1_run1000', 'low-accuracy')):
        g = load_golden('philox_%s.npz' % tag)
        imu = imu_model.IMU(accuracy=grade, axis=6, gps=False)
        for key, mine in (('gyro_b', imu.gyro_err['b']), ('gyro_b_drift', imu.gyro_err['b_drift']),
                          ('gyro_b_corr', imu.gyro_err['b_corr']), ('gyro_arw', imu.gyro_err['arw']),
                          ('accel_b', imu.accel_err['b']), ('accel_b_drift', imu.accel_err['b_drift']),
                          ('accel_b_corr', imu.accel_err['b_corr']), ('accel_vrw', imu.accel_err['vrw'])):
            assert np.array_equal(mine, g[key]), (grade, key)


def test_imu_custom_dict_units_and_errors():
    from gnss_ins_sim_b200 import imu_model
    d2r = np.pi / 180
    acc = {'gyro_b': np.array([1.0, 2.0, 3.0]), 'gyro_arw': np.array([0.25, 0.25, 0.25]),
           'gyro_b_stability': np.array([3.5, 3.5, 3.5]), 'gyro_b_corr': np.array([100.0] * 3),
           'accel_b': np.array([1e-3, 0, 0]), 'accel_vrw': np.array([0.03, 0.03, 0.04]),
           'accel_b_stability': np.array([4e-5, 5e-5, 8e-5])}
    imu = imu_model.IMU(accuracy=acc, axis=6, gps=False, odo=True, odo_opt={'scale': 0.999, 'stdv': 0.1})
    assert_close(imu.gyro_err['b'], acc['gyro_b'] * d2r / 3600, 1e-15, 0.0)
    assert_close(imu.gyro_err['arw'], acc['gyro_arw'] * d2r / 60, 1e-15, 0.0)
    assert_close(imu.accel_err['vrw'], acc['accel_vrw'] / 60, 1e-15, 0.0)
    assert np.isinf(imu.accel_err['b_corr']).all()          # missing corr time -> white drift
    assert imu.odo and imu.odo_err['scale'] == 0.999 and imu.gps is False and imu.gps_err is None
    other = imu_model.IMU(accuracy='low-accuracy', axis=6)   # no shared state (reference quirk)
    assert other.gyro_err['b_drift'][0] == 10.0 * d2r / 3600 and other.gps_err['stdp'][2] == 7.0
    with pytest.raises(ValueError):
        imu_model.IMU(axis=7)
    with pytest.raises(ValueError):
        imu_model.IMU(accuracy='best')
    with pytest.raises(ValueError):
        imu_model.IMU(accuracy={'gyro_b': 0})
    with pytest.raises(TypeError):
        imu_model.IMU(accuracy=3)
    with pytest.raises(ValueError):
        imu_model.IMU(accuracy=acc, axis=9)                  # magnetometer without mag_std
    with pytest.raises(ValueError):
        imu_model.IMU(gps=True, gps_opt={'stdp': 1})
    with pytest.raises(TypeError):
        imu_model.IMU(odo=True, odo_opt=3)
    imu.set_gyro_error('high-accuracy')
    assert imu.gyro_err['arw'][0] == 2.0e-3 * d2r / 60
    imu.set_accel_error({'vrw': np.ones(3)})
    assert imu.accel_err['vrw'][1] == 1.0
    with pytest.raises(ValueError):
        imu.set_accel_error({'nope': 1})


# ------------------------------------------------------------------ Sim host logic
def test_parse_env_matches_reference_dsl():
    from gnss_ins_sim_b200.sim import parse_env
    g = load_golden('philox_90deg_mid_rf1_vibrand.npz')
    a = parse_env('[0.03 0.001 0.01]-random', 100.0)
    assert a['type'] == 'random' and np.allclose([a['x'], a['y'], a['z']], g['vib_acc_amp'], rtol=0, atol=0)
    b = parse_env('[6 5 4]d-random', 100.0)
    assert np.array_equal([b['x'], b['y'], b['z']], g['vib_gyro_amp'])
    g = load_golden('philox_90deg_mid_rf0_vibsin.npz')
    c = parse_env('[0.03 0.001 0.01]g-3Hz-sinusoidal', 100.0)
    assert c['type'] == 'sinusoidal' and c['freq'] == 3.0
    assert np.array_equal([c['x'], c['y'], c['z']], g['vib_acc_amp'])
    d = parse_env('[6 5 4]d-0.5Hz-sinusoidal', 100.0)
    assert d['freq'] == 0.5 and np.array_equal([d['x'], d['y'], d['z']], g['vib_gyro_amp'])
    psd = np.array([[0.0, 1, 1, 1], [10.0, 2, 2, 2], [60.0, 3, 3, 3]])
    e = parse_env(psd, 100.0)
    assert e['type'] == 'psd' and len(e['freq']) == 2
    for bad in ('[1 2 3]-noise', '[1 2 3]-sinusoidal', '[a b c]-random'):
        with pytest.raises(ValueError):
            parse_env(bad, 100.0)
    with pytest.raises(TypeError):
        parse_env(3, 100.0)
    assert parse_env(None, 100.0) is None


def test_plugin_protocol_and_ini_sets():
    from gnss_ins_sim_b200.free_integration import FreeIntegration
    from gnss_ins_sim_b200.allan_analysis import Allan
    a = FreeIntegration(np.arange(9.0))
    assert a.input == ['ref_frame', 'fs', 'gyro', 'accel'] and a.output == ['att_euler', 'pos', 'vel']
    assert a.batch is True and a.set_of_inis == 1 and a.run_times == 0 and a.get_results() is None
    b = FreeIntegration(np.arange(30.0).reshape(10, 3), earth_rot=False)
    assert b.set_of_inis == 3 and b.ini_sets.shape == (3, 10) and b.ini_sets[1, 9] == 28.0
    with pytest.raises(ValueError):
        FreeIntegration(np.zeros((9, 2, 2)))
    with pytest.raises(ValueError):
        FreeIntegration(np.zeros(8))
    al = Allan()
    assert al.input == ['fs', 'accel', 'gyro'] and al.output == ['algo_time', 'ad_accel', 'ad_gyro']
    a.reset()
    al.reset()


def test_sim_validates_like_the_reference():
    from gnss_ins_sim_b200.sim import Sim, load_trajectory

    class Bad(object):
        input = []
        output = ['x']
    with pytest.raises(ValueError):
        Sim([100.0, 0, 0], {}, algorithm=Bad())
    t = load_trajectory(os.path.join(ROOT, 'tests', 'golden', 'traj_90deg_turn_100hz_rf1.npz'))
    assert t['ref_gyro'].shape == (1000, 3) and 'time' in t
    with pytest.raises(ValueError):
        load_trajectory({'ref_pos': np.zeros((3, 3))})
    s = Sim([100.0, 0, 0], t, ref_frame=7)
    assert s.ref_frame == 0 and s.results() is None         # run() first


# ------------------------------------------------------------------ multi-rank ---
def test_shard_partition():
    from gnss_ins_sim_b200 import dist
    for total in (0, 1, 7, 1000, 100000, 12345):
        for w in (1, 2, 3, 8):
            blocks = [dist.shard(total, r, w) for r in range(w)]
            assert blocks[0][0] == 0 and blocks[-1][1] == total
            assert all(blocks[i][1] == blocks[i + 1][0] for i in range(w - 1))
            sizes = [hi - lo for lo, hi in blocks]
            assert max(sizes) - min(sizes) <= 1


def test_merge_stats_is_as_good_as_two_pass():
    from gnss_ins_sim_b200 import dist
    rng = np.random.RandomState(1)
    x = rng.randn(1000, 9) * 1e-3 + 1e3          # mean >> std: one-pass sum-of-squares would fail
    cuts = [0, 1, 1, 400, 401, 1000]              # includes an empty shard and a 1-run shard
    blocks = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        part = x[a:b]
        blocks.append((b - a, np.abs(part).max(0) if b > a else np.zeros(9),
                       part.mean(0) if b > a else np.zeros(9), part.std(0) if b > a else np.zeros(9)))
    merged, n = dist.merge_stats(blocks)
    assert n == 1000
    assert_close(merged[1], x.mean(0), 1e-14, 0.0, 'mean')
    assert_close(merged[2], x.std(0), 1e-10, 0.0, 'std')
    assert np.array_equal(merged[0], np.abs(x).max(0))


def _gloo_worker(rank, world, port, tmp):
    import torch
    import torch.distributed as td
    sys.path.insert(0, ROOT)
    from gnss_ins_sim_b200 import dist
    td.init_process_group('gloo', init_method='tcp://127.0.0.1:%d' % port, rank=rank, world_size=world)
    rng = np.random.RandomState(0)
    total = 1001
    err = rng.randn(total, 9) * np.logspace(-4, 2, 9) + 0.3
    lo, hi = dist.shard(total)
    mine = torch.from_numpy(err[lo:hi])
    # what K3 phase 1 / 2 compute on each rank (numpy stands in for the kernels here)
    partial = torch.cat([mine.sum(0), mine.abs().max(0).values])
    mean, mx, tot = dist.combine_phase1(partial, hi - lo, 9)
    std = dist.combine_phase2(((mine - mean) ** 2).sum(0), tot)
    loc = mine.numpy()
    merged = dist.combine_local_stats(np.stack([np.abs(loc).max(0), loc.mean(0), loc.std(0)]), hi - lo)
    rows = dist.gather_rows(mine, total)
    traj = None
    if rank == 0:
        traj = {k: rng.randn(50, 3) for k in ('ref_pos', 'ref_vel', 'ref_att', 'ref_accel', 'ref_gyro')}
    got = dist.broadcast_trajectory(traj)
    np.savez(os.path.join(tmp, 'r%d.npz' % rank), mean=mean.numpy(), mx=mx.numpy(), std=std.numpy(),
             tot=tot, rows=rows, gyro=got['ref_gyro'], lo=lo, hi=hi, merged=merged)
    td.destroy_process_group()


def test_two_rank_statistics_over_gloo(tmp_path):
    import torch.multiprocessing as mp
    port = 29500 + (os.getpid() % 2000)
    mp.spawn(_gloo_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    rng = np.random.RandomState(0)
    err = rng.randn(1001, 9) * np.logspace(-4, 2, 9) + 0.3
    gyro0 = None
    for r in range(2):
        z = np.load(os.path.join(str(tmp_path), 'r%d.npz' % r))
        assert int(z['tot']) == 1001
        assert_close(z['mean'], err.mean(0), 1e-12, 1e-12, 'mean')
        assert_close(z['mx'], np.abs(err).max(0), 0.0, 0.0, 'max')
        assert_close(z['std'], err.std(0), 1e-12, 0.0, 'std')
        assert np.array_equal(z['rows'], err)
        assert_close(z['merged'], np.stack([np.abs(err).max(0), err.mean(0), err.std(0)]), 1e-12, 1e-12,
                     'one-collective merge')
        gyro0 = z['gyro'] if gyro0 is None else gyro0
        assert np.array_equal(z['gyro'], gyro0) and z['gyro'].shape == (50, 3)


# ------------------------------------------------------------------ path_gen (host) ---
def test_path_gen_matches_reference_trajectories():
    """gnss_ins_sim_b200.pathgen.path_gen (C++ on the host) against rows and column checksums of
    the reference's pathgen.path_gen for three motion definitions (all five command types, GPS
    and odometer outputs, both frames, up to 193 036 samples)."""
    from gnss_ins_sim_b200 import pathgen as pg
    g = load_golden('pathgen.npz')
    for tag, name, gps, odo in (('3d', 'motion_def-3d.csv', True, True),
                                ('full', 'motion_def.csv', False, True),
                                ('long_drive', 'motion_def-long_drive.csv', True, False)):
        fs, rf = float(g[tag + '_fs']), int(g[tag + '_rf'])
        ini, cmd = pg.parse_motion(os.path.join(ROOT, 'tests', 'golden', name))
        cmd0 = cmd.copy()
        od = np.array([[1.0, fs], [1.0 if gps else -1.0, 10.0], [1.0 if odo else -1.0, fs]])
        r = pg.path_gen(ini, cmd, od, pg.HIGH_MOBILITY, rf)
        assert np.array_equal(cmd, cmd0)                      # inputs are not modified
        assert r['nav'].shape == (int(g[tag + '_n']), 10) and r['status'] is True
        idx = g[tag + '_idx']
        assert_close(r['imu'][idx], g[tag + '_imu'], 1e-12, 1e-3, 'imu rows')
        assert_close(r['nav'][idx], g[tag + '_nav'], 1e-13, 1e-3, 'nav rows')
        assert_close(r['imu'].sum(0), g[tag + '_imu_sum'], 1e-11, 1.0, 'imu checksum')
        assert_close(np.abs(r['nav']).sum(0), g[tag + '_nav_abs_sum'], 1e-12, 1.0, 'nav checksum')
        if gps:
            assert r['gps'].shape[0] == int(g[tag + '_gps_n'])
            assert_close(r['gps'][::max(1, (idx[1] - idx[0]) // 10)], g[tag + '_gps'], 1e-13, 1e-3, 'gps')
        if odo:
            assert_close(r['odo'][idx], g[tag + '_odo'], 1e-13, 1e-3, 'odo')


def test_path_gen_reproduces_the_bench_trajectory_and_errors():
    from gnss_ins_sim_b200 import pathgen as pg
    from gnss_ins_sim_b200.sim import trajectory_from_motion_def
    for rf in (0, 1):
        g = load_golden('traj_90deg_turn_100hz_rf%d.npz' % rf)
        t = trajectory_from_motion_def(100.0, os.path.join(ROOT, 'tests', 'golden', 'motion_def-90deg_turn.csv'),
                                       rf)
        for k in ('ref_pos', 'ref_vel', 'ref_att', 'ref_accel', 'ref_gyro', 'time'):
            assert_close(t[k], g[k], 1e-13, 1e-6, k)
        assert_close(t['ini'], g['ini'], 0.0, 0.0, 'ini')
    text = ('ini lat (deg),ini lon (deg),ini alt (m),vx,vy,vz,yaw,pitch,roll\n32,120,0,0,0,0,0,0,0\n'
            'command type,yaw,pitch,roll,vx,vy,vz,duration,GPS\n1,0,0,0,0,0,0,2,0\n')
    t = trajectory_from_motion_def(100.0, text, 0, mode=np.array([1.0, 30.0, 60.0]))
    assert t['ref_gyro'].shape == (200, 3)
    with pytest.raises(ValueError):
        pg.path_gen(np.zeros(9), np.array([[1, 0, 0, 0, 0, 0, 0, -1.0, 0]]),
                    np.array([[1.0, 100.0], [-1.0, 100.0], [-1.0, 100.0]]), pg.HIGH_MOBILITY)
    with pytest.raises(NotImplementedError):
        pg.path_gen(np.zeros(9), np.array([[1, 0, 0, 0, 0, 0, 0, 1.0, 0]]),
                    np.array([[1.0, 100.0], [-1.0, 100.0], [-1.0, 100.0]]), pg.HIGH_MOBILITY, magnet=True)
    with pytest.raises(TypeError):
        pg.parse_mode(np.zeros(4))


def test_logged_data_directory_loader(tmp_path):
    """The reference Sim's file input (ins_sim.py:434-451, :508-559; sim_data.py:187-260): names and
    keys from file names, units from the header row, conversion to internal units."""
    from conftest import write_logged_dir
    from gnss_ins_sim_b200 import logged
    assert logged.name_and_key('Accel-12.CSV') == ('accel', 12)
    assert logged.name_and_key('ref_pos.csv') == ('ref_pos', None)
    assert logged.name_and_key('gyro-a.csv') == ('gyro', 'a')
    assert logged.name_and_key('ini.txt') == (None, None)
    g = load_golden('logged_bosch.npz')
    d = write_logged_dir(str(tmp_path / 'log'), g)
    assert logged.file_units(os.path.join(d, 'gyro-0.csv')) == ['deg/s'] * 3
    data = logged.read_data_dir(d, 0)
    assert sorted(data) == ['accel', 'gyro', 'ref_att_euler', 'ref_pos', 'ref_vel', 'time']
    assert_close(data['gyro'][0], g['gyro'], 1e-15, 1e-9, 'gyro deg/s -> rad/s')
    assert np.array_equal(data['accel'][0], g['accel'])
    assert data['time'].shape == (1000,)
    # an LLA position file in the virtual inertial frame becomes metres (ins_sim.py:809-825)
    lla = np.array([[32.0, 120.0, 5.0], [32.00001, 120.00002, 6.0]])
    xyz, units = logged.convert_pos(lla, ['deg', 'deg', 'm'], 1)
    assert units == ['m', 'm', 'm']
    ecef = onp.lla2ecef(lla * np.array([np.pi / 180, np.pi / 180, 1.0]))
    assert_close(xyz[0], ecef[0], 1e-15, 1.0, 'first sample = its ECEF position')
    assert abs(np.linalg.norm(xyz[1] - xyz[0]) - np.linalg.norm(ecef[1] - ecef[0])) < 1e-9
    assert_close(logged.convert_units(np.array([[3600.0, 1.0, 2.0]]), ['deg/hr', 'rad/s', 'rad/s'],
                                      ['rad/s'] * 3), [[np.pi / 180, 1.0, 2.0]], 1e-15, 0.0, 'deg/hr')


def test_csv_files_round_trip(tmp_path):
    """write_data (Sim_data.save_to_file format: output units, legend header) -> read_data_dir."""
    from gnss_ins_sim_b200 import logged
    rng = np.random.RandomState(3)
    d = str(tmp_path / 'out')
    gyro = {0: rng.randn(50, 3) * 0.01, 1: rng.randn(50, 3) * 0.01}
    ref_pos = np.stack([0.55 + 1e-6 * rng.rand(50), 2.09 + 1e-6 * rng.rand(50), 10 * rng.rand(50)], 1)
    files = logged.write_data(d, 'gyro', gyro, 0) + logged.write_data(d, 'ref_pos', ref_pos, 0) \
        + logged.write_data(d, 'time', np.arange(50) / 100.0, 0)
    assert sorted(os.path.basename(f) for f in files) == ['gyro-0.csv', 'gyro-1.csv', 'ref_pos.csv', 'time.csv']
    assert open(files[0]).readline().strip() == 'gyro_x (deg/s),gyro_y (deg/s),gyro_z (deg/s)'
    assert open(files[2]).readline().strip() == 'ref_pos_lat (deg),ref_pos_lon (deg),ref_pos_alt (m)'
    back = logged.read_data_dir(d, 0)
    assert_close(back['gyro'][1], gyro[1], 1e-15, 1e-18, 'gyro')
    assert_close(back['ref_pos'], ref_pos, 1e-15, 0.0, 'ref_pos')
    assert_close(back['time'], np.arange(50) / 100.0, 1e-15, 0.0, 'time')
    # virtual inertial frame: positions are metres and stay as they are
    xyz = rng.randn(50, 3) * 1e6
    logged.write_data(d + '1', 'ref_pos', xyz, 1)
    assert open(os.path.join(d + '1', 'ref_pos.csv')).readline().strip() == 'ref_pos_x (m),ref_pos_y (m),ref_pos_z (m)'
    assert_close(logged.read_data_dir(d + '1', 1)['ref_pos'], xyz, 1e-15, 0.0, 'xyz')


def test_lanes_per_run_choice():
    """lanes_per_run = 0: the narrowest lane group that still gives every SM a CTA of the
    warp-specialised kernel (32 / G runs per CTA), one lane per run for large ensembles; supplied data /
    process statistics keep the one-warp-per-sub-partition rule.  Pure host logic (148 SMs given
    explicitly)."""
    from gnss_ins_sim_b200 import _lib
    lib = _lib.load()
    pick = lambda runs, fused: lib.b2ins_diag_auto_lanes(runs, fused, 148)   # noqa: E731
    assert [pick(r, 1) for r in (100, 500, 592, 593, 1000, 1184, 1185, 2000, 4000, 4736, 4737, 12500)] == \
        [8, 8, 8, 4, 4, 4, 2, 2, 2, 2, 1, 1]
    assert pick(40001, 1) == 1 and pick(10 ** 6, 1) == 1
    assert [pick(r, 0) for r in (500, 1000, 2000, 4000, 10000, 20000, 10 ** 6)] == [32, 16, 8, 4, 2, 1, 1]
    assert _lib.mc_shape(4, 0) == '6,1,0' and _lib.mc_shape(4, 1) == '6,2,0' and _lib.mc_shape(32) == '1,4,1'
    # every choice is a width the kernels are instantiated for
    assert all(pick(r, f) in (1, 2, 4, 8, 16, 32) for r in range(1, 60000, 997) for f in (0, 1))
