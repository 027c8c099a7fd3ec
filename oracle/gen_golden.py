"""
Generate tests/golden/*.npz by running the UNMODIFIED reference (gnss-ins-sim,
imported from /root/reference) in this container.  Test infrastructure only.

    python oracle/gen_golden.py            # writes tests/golden/

What is frozen (SURVEY 8c):
  logged_{bosch,nxp}.npz    demo_free_integration_openimu.py semantics: logged IMU
                            data, ref_frame=0, earth_rot=False, gravity from ini.txt.
  seeded_90deg_rf{0,1}.npz  np.random.seed(12345); 'mid-accuracy'; run(2): the
                            reference's own gyro/accel and its att/pos/vel.
  philox_*.npz              the b2ins Philox normal stream (oracle_np.noise_normals)
                            injected into the reference's np.random.randn call
                            sequence; reference outputs + end-point error stats
                            (string profiles, random / sinusoidal / PSD vibration, a dict
                            IMU with white bias drift, the odometer variant).
  ned_stats_*.npz           get_error_stats('pos', extra_opt='ned'|'ecef') of the reference.
  traj_*.npz                pathgen.path_gen output (true trajectory + ideal IMU).
  allan.npz, psd.npz        allan.allan_var / time_series_from_psd known answers.

The reference cannot travel to the GPU box, the .npz files do.
"""
import math
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get('B2INS_REFERENCE', '/root/reference')
sys.path.insert(0, REF)
sys.path.insert(0, HERE)

from gnss_ins_sim.sim import ins_sim, imu_model          # noqa: E402
from gnss_ins_sim.pathgen import pathgen                  # noqa: E402
from gnss_ins_sim.allan import allan                      # noqa: E402
from gnss_ins_sim.psd import time_series_from_psd as ref_psd   # noqa: E402
from demo_algorithms import free_integration              # noqa: E402
import oracle_np as onp                                   # noqa: E402

D2R = math.pi / 180
OUT = os.path.join(os.path.dirname(HERE), 'tests', 'golden')
MOTION = os.path.join(REF, 'demo_motion_def_files')


class RandnQueue:
    """Stand-in for np.random.randn serving prepared arrays in call order."""

    def __init__(self):
        self.q = []
        self.calls = []

    def push(self, arr):
        self.q.append(np.array(arr, dtype=np.float64))

    def __call__(self, *shape):
        self.calls.append(shape)
        a = self.q.pop(0)
        assert a.shape == tuple(shape), (a.shape, shape)
        return a


def read_ini(path_csv):
    ini = np.genfromtxt(path_csv, delimiter=',', skip_header=1, max_rows=1)
    ini[0] *= D2R
    ini[1] *= D2R
    ini[6:9] *= D2R
    return ini


def fresh_imu(accuracy):
    # imu_model.IMU mutates module-level dicts when given a dict (SURVEY 7 quirks);
    # only the string profiles are used here, which are read-only.
    return imu_model.IMU(accuracy=accuracy, axis=6, gps=False)


def err_dict(e, white_key):
    return {'b': np.array(e['b']), 'b_drift': np.array(e['b_drift']),
            'b_corr': np.array(e['b_corr']), white_key: np.array(e[white_key])}


def collect(sim, R):
    d = sim.dmgr
    out = {
        'time': d.time.data, 'ref_pos': d.ref_pos.data, 'ref_vel': d.ref_vel.data,
        'ref_att': d.ref_att_euler.data, 'ref_accel': d.ref_accel.data,
        'ref_gyro': d.ref_gyro.data,
        'gyro': np.stack([d.gyro.data[i] for i in range(R)]),
        'accel': np.stack([d.accel.data[i] for i in range(R)]),
        'att': np.stack([d.att_euler.data['algo0_%d' % i] for i in range(R)]),
        'pos': np.stack([d.pos.data['algo0_%d' % i] for i in range(R)]),
        'vel': np.stack([d.vel.data['algo0_%d' % i] for i in range(R)]),
    }
    for name, ang in (('att_euler', True), ('pos', False), ('vel', False)):
        st = d.get_error_stats(name, err_stats_start=-1, angle=ang, use_output_units=False)
        for k in ('max', 'avg', 'std'):
            out['stat_%s_%s' % (name, k)] = np.asarray(st[k])
    return out


def gen_logged(name):
    log_dir = os.path.join(REF, 'demo_data_files', name) + '/'
    ini = np.genfromtxt(log_dir + 'ini.txt', delimiter=',')
    ini[0:2] *= D2R
    ini[6:9] *= D2R
    algo = free_integration.FreeIntegration(ini, earth_rot=False)
    sim = ins_sim.Sim([100.0, 0.0, 0.0], log_dir, ref_frame=0, imu=None, algorithm=algo)
    sim.run(1)
    d = sim.dmgr
    np.savez_compressed(os.path.join(OUT, 'logged_%s.npz' % name),
                        fs=100.0, ref_frame=0, earth_rot=False, ini=ini,
                        gyro=d.gyro.data[0], accel=d.accel.data[0],
                        att=d.att_euler.data['algo0_0'], pos=d.pos.data['algo0_0'],
                        vel=d.vel.data['algo0_0'])


def gen_seeded(ref_frame):
    csv = os.path.join(MOTION, 'motion_def-90deg_turn.csv')
    ini = read_ini(csv)
    np.random.seed(12345)
    imu = fresh_imu('mid-accuracy')
    algo = free_integration.FreeIntegration(ini)
    sim = ins_sim.Sim([100.0, 0.0, 0.0], csv, ref_frame=ref_frame, imu=imu, algorithm=algo)
    sim.run(2)
    out = collect(sim, 2)
    np.savez_compressed(os.path.join(OUT, 'seeded_90deg_rf%d.npz' % ref_frame),
                        fs=100.0, ref_frame=ref_frame, ini=ini, **out)


def inject_stream(q, n, run_ids, seed, vib_acc=None, vib_gyro=None):
    """Queue the b2ins normals in the reference's call order (SURVEY 3.3):
    per run: acc GM x3 (n,3) [column i used], [acc vib x3 (n,)], acc white (n,3),
             gyro GM x3, [gyro vib x3], gyro white."""
    z = onp.noise_normals(n, run_ids, seed)
    zva, zvg = onp.vib_normals(n, run_ids, seed)
    for r in range(len(run_ids)):
        for gm, w, vib, zv in ((z['acc_gm'], z['acc_w'], vib_acc, zva),
                               (z['gyr_gm'], z['gyr_w'], vib_gyro, zvg)):
            for i in range(3):
                blk = np.full((n, 3), np.nan)     # unused entries must never matter
                blk[:, i] = gm[r, :, i]
                q.push(blk)
            if vib is not None and vib['type'] == 'random':
                for i in range(3):
                    q.push(zv[r, :, i])
            q.push(w[r])


def gen_philox(tag, motion, fs, accuracy, ref_frame, R, seed, env=None, run0=0):
    csv = os.path.join(MOTION, motion)
    ini = read_ini(csv)
    imu = fresh_imu(accuracy)
    algo = free_integration.FreeIntegration(ini)
    sim = ins_sim.Sim([fs, 0.0, 0.0], csv, ref_frame=ref_frame, imu=imu, env=env,
                      algorithm=algo)
    # trajectory length is needed before the stream can be queued: run path_gen the
    # way Sim does (it is deterministic), then run Sim with the queue installed.
    probe = ins_sim.Sim([fs, 0.0, 0.0], csv, ref_frame=ref_frame, imu=imu, algorithm=None)
    real_randn, real_rand = np.random.randn, np.random.rand
    np.random.randn = lambda *s: np.zeros(s)
    try:
        probe.run(1)
    finally:
        np.random.randn = real_randn
    n = probe.dmgr.time.data.shape[0]
    run_ids = np.arange(run0, run0 + R)
    vib_acc = vib_gyro = None
    if env is not None:
        vib_acc = sim._Sim__parse_env(env['acc']) if 'acc' in env else None
        vib_gyro = sim._Sim__parse_env(env['gyro']) if 'gyro' in env else None
    q = RandnQueue()
    inject_stream(q, n, run_ids, seed, vib_acc, vib_gyro)
    phases = onp.gyro_vib_phase_uniforms(run_ids, seed)
    pq = [phases[r, c] for r in range(R) for c in range(3)]
    np.random.randn = q
    np.random.rand = lambda *s: np.array([pq.pop(0)])
    try:
        sim.run(R)
    finally:
        np.random.randn, np.random.rand = real_randn, real_rand
    assert not q.q, 'unused queued normals: %d' % len(q.q)
    out = collect(sim, R)
    extra = {}
    if env is not None:
        for k, v in (('vib_acc', vib_acc), ('vib_gyro', vib_gyro)):
            if v is not None:
                extra[k + '_type'] = v['type']
                extra[k + '_amp'] = np.array([v['x'], v['y'], v['z']])
                extra[k + '_freq'] = v.get('freq', 0.0)
    np.savez_compressed(os.path.join(OUT, 'philox_%s.npz' % tag),
                        fs=fs, ref_frame=ref_frame, ini=ini, seed=seed, run_ids=run_ids,
                        accuracy=accuracy,
                        gyro_b=imu.gyro_err['b'], gyro_b_drift=imu.gyro_err['b_drift'],
                        gyro_b_corr=imu.gyro_err['b_corr'], gyro_arw=imu.gyro_err['arw'],
                        accel_b=imu.accel_err['b'], accel_b_drift=imu.accel_err['b_drift'],
                        accel_b_corr=imu.accel_err['b_corr'], accel_vrw=imu.accel_err['vrw'],
                        **out, **extra)


def gen_philox_config3(R=2, seed=11, stride=2000):
    """BASELINE config 3 at its FULL length through the unmodified reference: motion_def-long_drive.csv
    @200 Hz (193 036 samples), 'low-accuracy' IMU, ref_frame 0, R runs on the b2ins stream (run ids
    0..R-1, as Sim(seed=...).run(R) names them).  Kept: the end-point state and error of every run and
    the histories at every `stride`-th sample (the full arrays are 14 MB per run)."""
    csv = os.path.join(MOTION, 'motion_def-long_drive.csv')
    ini = read_ini(csv)
    imu = fresh_imu('low-accuracy')
    fs = 200.0
    algo = free_integration.FreeIntegration(ini)
    sim = ins_sim.Sim([fs, 0.0, 0.0], csv, ref_frame=0, imu=imu, algorithm=algo)
    probe = ins_sim.Sim([fs, 0.0, 0.0], csv, ref_frame=0, imu=imu, algorithm=None)
    real_randn, real_rand = np.random.randn, np.random.rand
    np.random.randn = lambda *s: np.zeros(s)
    try:
        probe.run(1)
    finally:
        np.random.randn = real_randn
    n = probe.dmgr.time.data.shape[0]
    run_ids = np.arange(R)
    q = RandnQueue()
    inject_stream(q, n, run_ids, seed)
    np.random.randn = q
    try:
        sim.run(R)
    finally:
        np.random.randn, np.random.rand = real_randn, real_rand
    assert not q.q, 'unused queued normals: %d' % len(q.q)
    d = sim.dmgr
    att = np.stack([d.att_euler.data['algo0_%d' % i] for i in range(R)])
    pos = np.stack([d.pos.data['algo0_%d' % i] for i in range(R)])
    vel = np.stack([d.vel.data['algo0_%d' % i] for i in range(R)])
    end_state = np.concatenate([att[:, -1], pos[:, -1], vel[:, -1]], axis=1)
    ref_end = np.concatenate([d.ref_att_euler.data[-1], d.ref_pos.data[-1], d.ref_vel.data[-1]])
    np.savez_compressed(os.path.join(OUT, 'philox_config3_long_drive_rf0.npz'),
                        fs=fs, n=n, seed=seed, run_ids=run_ids, ini=ini, stride=stride,
                        end_state=end_state, ref_end=ref_end,
                        att=att[:, ::stride], pos=pos[:, ::stride], vel=vel[:, ::stride],
                        ref_pos=d.ref_pos.data[::stride], ref_att=d.ref_att_euler.data[::stride])


def gen_ned_stats(R=8, seed=12345):
    """get_error_stats('pos', extra_opt='ned' | 'ecef') of the reference (ins_data_manager.py:543-552)
    for the philox_90deg_mid_rf0 experiment: LLA end-point errors in metres, in the local NED frame or
    in ECEF.  The reference caches the error array of a data name at the first call
    (ins_data_manager.py:427-431), so a second call with another option would return the first
    option's numbers: every option gets a fresh Sim (first-call behaviour is what is frozen)."""
    csv = os.path.join(MOTION, 'motion_def-90deg_turn.csv')
    ini = read_ini(csv)
    n, run_ids = 1000, np.arange(R)
    out = {'seed': seed, 'run_ids': run_ids}
    g = np.load(os.path.join(OUT, 'philox_90deg_mid_rf0.npz'))
    for opt in ('ned', 'ecef'):
        imu = fresh_imu('mid-accuracy')
        sim = ins_sim.Sim([100.0, 0.0, 0.0], csv, ref_frame=0, imu=imu,
                          algorithm=free_integration.FreeIntegration(ini))
        q = RandnQueue()
        inject_stream(q, n, run_ids, seed)
        real = np.random.randn
        np.random.randn = q
        try:
            sim.run(R)
        finally:
            np.random.randn = real
        assert not q.q
        # the run must be the one frozen in philox_90deg_mid_rf0.npz
        assert np.array_equal(g['pos'][3], sim.dmgr.pos.data['algo0_3'])
        st = sim.dmgr.get_error_stats('pos', err_stats_start=-1, angle=False, use_output_units=False,
                                      extra_opt=opt)
        for k in ('max', 'avg', 'std'):
            out['stat_pos_%s_%s' % (opt, k)] = np.asarray(st[k])
    assert not np.allclose(out['stat_pos_ned_std'], out['stat_pos_ecef_std'])
    np.savez_compressed(os.path.join(OUT, 'ned_stats_90deg_mid_rf0.npz'), **out)


def gen_philox_white_drift(ref_frame, R=4, seed=31337):
    """A dict-`accuracy` IMU without *_b_corr: the bias drift is white, drift[i]*randn(n) per axis
    (pathgen.py:591-593) -- three (n,) draws per sensor instead of three (n,3) blocks; they are served
    the GM-drive normals of the b2ins stream.  (The dict form writes into the module-level
    'low-accuracy' tables, imu_model.py:110-143: restored afterwards.)"""
    import copy
    csv = os.path.join(MOTION, 'motion_def-90deg_turn.csv')
    ini = read_ini(csv)
    saved = copy.deepcopy((imu_model.gyro_low_accuracy, imu_model.accel_low_accuracy))
    acc = {'gyro_b': np.array([36.0, -20.0, 5.0]), 'gyro_arw': np.array([0.3, 0.25, 0.2]),
           'gyro_b_stability': np.array([8.0, 6.0, 4.0]),
           'accel_b': np.array([1e-3, -2e-3, 5e-4]), 'accel_vrw': np.array([0.04, 0.03, 0.05]),
           'accel_b_stability': np.array([1e-4, 2e-4, 5e-5])}
    try:
        imu = imu_model.IMU(accuracy=acc, axis=6, gps=False)
        assert np.all(np.isinf(imu.gyro_err['b_corr'])) and np.all(np.isinf(imu.accel_err['b_corr']))
        errs = {k: np.array(v) for k, v in (
            ('gyro_b', imu.gyro_err['b']), ('gyro_b_drift', imu.gyro_err['b_drift']),
            ('gyro_b_corr', imu.gyro_err['b_corr']), ('gyro_arw', imu.gyro_err['arw']),
            ('accel_b', imu.accel_err['b']), ('accel_b_drift', imu.accel_err['b_drift']),
            ('accel_b_corr', imu.accel_err['b_corr']), ('accel_vrw', imu.accel_err['vrw']))}
        sim = ins_sim.Sim([100.0, 0.0, 0.0], csv, ref_frame=ref_frame, imu=imu,
                          algorithm=free_integration.FreeIntegration(ini))
        n, run_ids = 1000, np.arange(R) + 2
        z = onp.noise_normals(n, run_ids, seed)
        q = RandnQueue()
        for r in range(R):
            for gm, w in ((z['acc_gm'], z['acc_w']), (z['gyr_gm'], z['gyr_w'])):
                for i in range(3):
                    q.push(gm[r, :, i])          # drift[i] * randn(n)
                q.push(w[r])
        real = np.random.randn
        np.random.randn = q
        try:
            sim.run(R)
        finally:
            np.random.randn = real
        assert not q.q
        out = collect(sim, R)
    finally:
        imu_model.gyro_low_accuracy.clear()
        imu_model.gyro_low_accuracy.update(saved[0])
        imu_model.accel_low_accuracy.clear()
        imu_model.accel_low_accuracy.update(saved[1])
    np.savez_compressed(os.path.join(OUT, 'philox_90deg_whitedrift_rf%d.npz' % ref_frame), fs=100.0,
                        ref_frame=ref_frame, ini=ini, seed=seed, run_ids=run_ids,
                        **{'acc_' + k: v for k, v in acc.items()}, **errs, **out)


def gen_philox_psd(ref_frame=1, R=3, seed=606):
    """PSD vibration through the reference Sim: env = {'acc': table, 'gyro': table} (n,4) arrays
    (ins_sim.py:642-701); acc_gen / gyro_gen call time_series_from_psd per axis after the bias-drift
    blocks (pathgen.py:478-485, :541-548), each drawing randn(L) random phases -- served from the
    b2ins stream (draws 16 + 3*sensor + axis)."""
    csv = os.path.join(MOTION, 'motion_def-90deg_turn.csv')
    ini = read_ini(csv)
    tab = np.genfromtxt(os.path.join(MOTION, 'vib_psd.csv'), delimiter=',', skip_header=1)
    env_acc = tab.copy()
    env_gyro = tab.copy()
    env_gyro[:, 1:] *= 1e-4 * np.array([1.0, 0.5, 0.25])     # (rad/s)^2/Hz: a different table per axis
    imu = fresh_imu('mid-accuracy')
    sim = ins_sim.Sim([100.0, 0.0, 0.0], csv, ref_frame=ref_frame, imu=imu,
                      env={'acc': env_acc.copy(), 'gyro': env_gyro.copy()},
                      algorithm=free_integration.FreeIntegration(ini))
    n, run_ids = 1000, np.arange(R) + 10
    L = n // 2 + 1
    z = onp.noise_normals(n, run_ids, seed)
    zp = {0: onp.psd_phase_normals(L, run_ids, seed, 0), 1: onp.psd_phase_normals(L, run_ids, seed, 1)}
    q = RandnQueue()
    for r in range(R):
        for sensor, gm, w in ((0, z['acc_gm'], z['acc_w']), (1, z['gyr_gm'], z['gyr_w'])):
            for i in range(3):
                blk = np.full((n, 3), np.nan)
                blk[:, i] = gm[r, :, i]
                q.push(blk)
            for i in range(3):
                q.push(zp[sensor][r, i])
            q.push(w[r])
    real = np.random.randn
    np.random.randn = q
    try:
        sim.run(R)
    finally:
        np.random.randn = real
    assert not q.q
    out = collect(sim, R)
    np.savez_compressed(os.path.join(OUT, 'philox_90deg_mid_rf%d_psd.npz' % ref_frame), fs=100.0,
                        ref_frame=ref_frame, ini=ini, seed=seed, run_ids=run_ids, env_acc=env_acc,
                        env_gyro=env_gyro, **out)


def gen_philox_odo(ref_frame, R=6, seed=4711):
    """demo_free_integration.py semantics: IMU(odo=True), algorithm = free_integration_odo
    (demo_free_integration.py:40,61-71); the odometer draw (pathgen.py:639) is served from the
    b2ins stream after the gyro white block (ins_sim.py:503-506)."""
    from demo_algorithms import free_integration_odo
    csv = os.path.join(MOTION, 'motion_def-90deg_turn.csv')
    ini = read_ini(csv)
    odo_err = {'scale': 0.999, 'stdv': 0.1}
    imu = imu_model.IMU(accuracy='mid-accuracy', axis=6, gps=False, odo=True, odo_opt=odo_err)
    algo = free_integration_odo.FreeIntegration(ini)
    sim = ins_sim.Sim([100.0, 0.0, 0.0], csv, ref_frame=ref_frame, imu=imu, algorithm=algo)
    n = 1000
    run_ids = np.arange(R)
    z = onp.noise_normals(n, run_ids, seed)
    zo = onp.odo_normals(n, run_ids, seed)
    q = RandnQueue()
    for r in range(R):
        for gm, w in ((z['acc_gm'], z['acc_w']), (z['gyr_gm'], z['gyr_w'])):
            for i in range(3):
                blk = np.full((n, 3), np.nan)
                blk[:, i] = gm[r, :, i]
                q.push(blk)
            q.push(w[r])
        q.push(zo[r])
    real = np.random.randn
    np.random.randn = q
    try:
        sim.run(R)
    finally:
        np.random.randn = real
    assert not q.q
    d = sim.dmgr
    out = collect(sim, R)
    np.savez_compressed(os.path.join(OUT, 'philox_90deg_mid_rf%d_odo.npz' % ref_frame),
                        fs=100.0, ref_frame=ref_frame, ini=ini, seed=seed, run_ids=run_ids,
                        odo_scale=odo_err['scale'], odo_stdv=odo_err['stdv'],
                        ref_odo=d.ref_odo.data, odo=np.stack([d.odo.data[i] for i in range(R)]),
                        gyro_b=imu.gyro_err['b'], gyro_b_drift=imu.gyro_err['b_drift'],
                        gyro_b_corr=imu.gyro_err['b_corr'], gyro_arw=imu.gyro_err['arw'],
                        accel_b=imu.accel_err['b'], accel_b_drift=imu.accel_err['b_drift'],
                        accel_b_corr=imu.accel_err['b_corr'], accel_vrw=imu.accel_err['vrw'], **out)


def gen_gps(ref_frame, R=4, seed=2024):
    """IMU(gps=True) at 10 Hz: after the 8 IMU blocks of a run the reference draws the GPS position
    and velocity noise, two (m, 3) blocks (pathgen.py:622-623 via ins_sim.py:497-500); they are
    served from the b2ins stream (draws 24..26)."""
    csv = os.path.join(MOTION, 'motion_def-90deg_turn.csv')
    gps_err = {'stdp': np.array([5.0, 5.0, 7.0]), 'stdv': np.array([0.05, 0.05, 0.05])}
    imu = imu_model.IMU(accuracy='mid-accuracy', axis=6, gps=True, gps_opt=gps_err)
    sim = ins_sim.Sim([100.0, 10.0, 0.0], csv, ref_frame=ref_frame, imu=imu, algorithm=None)
    n, m = 1000, 100
    run_ids = np.arange(R) + 5
    z = onp.noise_normals(n, run_ids, seed)
    zg = onp.gps_normals(m, run_ids, seed)
    q = RandnQueue()
    for r in range(R):
        for gm, w in ((z['acc_gm'], z['acc_w']), (z['gyr_gm'], z['gyr_w'])):
            for i in range(3):
                blk = np.full((n, 3), np.nan)
                blk[:, i] = gm[r, :, i]
                q.push(blk)
            q.push(w[r])
        q.push(zg[r, :, 0:3])
        q.push(zg[r, :, 3:6])
    real = np.random.randn
    np.random.randn = q
    try:
        sim.run(R)
    finally:
        np.random.randn = real
    assert not q.q
    d = sim.dmgr
    assert d.ref_gps.data.shape == (m, 6)
    np.savez_compressed(os.path.join(OUT, 'gps_90deg_rf%d.npz' % ref_frame),
                        ref_frame=ref_frame, seed=seed, run_ids=run_ids, stdp=gps_err['stdp'],
                        stdv=gps_err['stdv'], ref_gps=d.ref_gps.data, gps_time=d.gps_time.data,
                        gps_visibility=d.gps_visibility.data,
                        gps=np.stack([d.gps.data[i] for i in range(R)]))


def gen_traj(tag, motion, fs, ref_frame):
    csv = os.path.join(MOTION, motion)
    imu = fresh_imu('low-accuracy')
    sim = ins_sim.Sim([fs, 0.0, 0.0], csv, ref_frame=ref_frame, imu=imu, algorithm=None)
    real = np.random.randn
    np.random.randn = lambda *s: np.zeros(s)
    try:
        sim.run(1)
    finally:
        np.random.randn = real
    d = sim.dmgr
    np.savez_compressed(os.path.join(OUT, 'traj_%s.npz' % tag), fs=fs, ref_frame=ref_frame,
                        ini=read_ini(csv), time=d.time.data, ref_pos=d.ref_pos.data,
                        ref_vel=d.ref_vel.data, ref_att=d.ref_att_euler.data,
                        ref_accel=d.ref_accel.data, ref_gyro=d.ref_gyro.data)


def gen_pathgen():
    """pathgen.path_gen outputs (strided rows + column checksums) for three motion definitions,
    and the motion-definition files themselves as input fixtures (tests/golden/motion_def*.csv)."""
    import shutil
    out = {}
    for tag, name, fs, rf, gps, odo, stride in (('3d', 'motion_def-3d.csv', 100.0, 0, True, True, 7),
                                                ('full', 'motion_def.csv', 50.0, 1, False, True, 31),
                                                ('long_drive', 'motion_def-long_drive.csv', 200.0, 0,
                                                 True, False, 997)):
        shutil.copy(os.path.join(MOTION, name), os.path.join(OUT, name))
        sim = ins_sim.Sim([fs, 10.0, 0.0], os.path.join(MOTION, name), ref_frame=rf,
                          imu=fresh_imu('low-accuracy'), algorithm=None)
        ini, cmd = sim._Sim__parse_motion()
        od = np.array([[1.0, fs], [1.0 if gps else -1.0, 10.0], [1.0 if odo else -1.0, fs]])
        r = pathgen.path_gen(ini, cmd, od, np.array([1.0, 0.5, 2.0]), rf, False)
        n = r['nav'].shape[0]
        idx = np.unique(np.concatenate([np.arange(0, n, stride), [n - 1]]))
        out.update({tag + '_n': n, tag + '_idx': idx, tag + '_fs': fs, tag + '_rf': rf,
                    tag + '_imu': r['imu'][idx], tag + '_nav': r['nav'][idx],
                    tag + '_imu_sum': r['imu'].sum(0), tag + '_nav_abs_sum': np.abs(r['nav']).sum(0)})
        if gps:
            out[tag + '_gps'] = r['gps'][::max(1, stride // 10)]
            out[tag + '_gps_n'] = r['gps'].shape[0]
        if odo:
            out[tag + '_odo'] = r['odo'][idx]
    shutil.copy(os.path.join(MOTION, 'motion_def-90deg_turn.csv'), os.path.join(OUT, 'motion_def-90deg_turn.csv'))
    np.savez_compressed(os.path.join(OUT, 'pathgen.npz'), **out)


def gen_allan():
    seed = 2024
    rng = np.random.RandomState(seed)
    fs = 100.0
    n = 180000
    # white + random walk + a GM-like component: exercises all tau decades
    # (tests/conftest.py:allan_golden regenerates x from the seed: the series alone is 1.4 MB)
    x = 0.01 * rng.randn(n) + np.cumsum(1e-5 * rng.randn(n))
    avar, tau = allan.allan_var(x, fs)
    x2 = rng.randn(7351)       # ragged: n not a multiple of anything
    avar2, tau2 = allan.allan_var(x2, 50.0)
    x3 = rng.randn(800)        # too short: max_bin*ts < 1 -> ([], [])
    a3, t3 = allan.allan_var(x3, 100.0)
    assert len(a3) == 0
    np.savez_compressed(os.path.join(OUT, 'allan.npz'), fs=fs, seed=seed, n=n, x_every_1000=x[::1000],
                        avar=avar, tau=tau, fs2=50.0, x2=x2, avar2=avar2, tau2=tau2, x3=x3)


def gen_allan_config4(n=14400000, fs=400.0, seed=5, run=2):
    """BASELINE config 4 at its FULL length: allan.allan_var of the unmodified reference on ONE 14.4 M-sample
    series (10 h @400 Hz): the gyro-z and accel-x measurements of run `run` of a static 'low-accuracy' IMU
    on the b2ins stream (made by the C oracle's generator -- any input would do, this is the one the
    config-4 tests already produce).  Kept: tau and the two Allan variances (55 values each)."""
    import oracle_c
    imu = fresh_imu('low-accuracy')
    ref_gyro = np.zeros((n, 3))
    ref_accel = np.tile(np.array([4.9, 0.0, -8.487]), (n, 1))        # 30 deg pitch, static
    og, oa = oracle_c.imu_noise(fs, ref_gyro, ref_accel, imu.gyro_err, imu.accel_err, seed, [run])
    avar_g, tau = allan.allan_var(np.ascontiguousarray(og[0, :, 2]), fs)
    avar_a, tau_a = allan.allan_var(np.ascontiguousarray(oa[0, :, 0]), fs)
    assert np.array_equal(tau, tau_a)
    np.savez_compressed(os.path.join(OUT, 'allan_config4_full_length.npz'), n=n, fs=fs, seed=seed, run=run,
                        tau=tau, avar_gyro_z=avar_g, avar_accel_x=avar_a)


def gen_psd():
    tab = np.genfromtxt(os.path.join(MOTION, 'vib_psd.csv'), delimiter=',', skip_header=1)
    rng = np.random.RandomState(7)
    out = {}
    for tag, fs, n in (('a', 200.0, 1000), ('b', 200.0, 40001)):
        half = 0.5 * fs
        m = tab.shape[0]
        if tab[-1, 0] > half:
            m = np.where(tab[:, 0] > half)[0][0]
        freq = tab[:m, 0].copy()
        sxx = tab[:m, 1].copy()
        N = n if n % 2 == 0 else n + 1
        N = min(N, 16384)
        L = N // 2 + 1
        zn = rng.randn(L)
        real = np.random.randn
        np.random.randn = lambda *s: zn.copy()
        try:
            ok, x = ref_psd.time_series_from_psd(sxx.copy(), freq, fs, n)
        finally:
            np.random.randn = real
        assert ok
        out.update({'freq_' + tag: freq, 'sxx_' + tag: sxx, 'fs_' + tag: fs, 'n_' + tag: n,
                    'z_' + tag: zn, 'x_' + tag: x})
    np.savez_compressed(os.path.join(OUT, 'psd.npz'), **out)


def main():
    os.makedirs(OUT, exist_ok=True)
    gen_logged('bosch')
    gen_logged('nxp')
    gen_seeded(0)
    gen_seeded(1)
    gen_philox('90deg_mid_rf1', 'motion_def-90deg_turn.csv', 100.0, 'mid-accuracy', 1, 8, 12345)
    gen_philox('90deg_mid_rf0', 'motion_def-90deg_turn.csv', 100.0, 'mid-accuracy', 0, 8, 12345)
    gen_philox('90deg_low_rf1_run1000', 'motion_def-90deg_turn.csv', 100.0, 'low-accuracy', 1, 4,
               987654321987, run0=1000)
    gen_philox('90deg_mid_rf1_vibrand', 'motion_def-90deg_turn.csv', 100.0, 'mid-accuracy', 1, 3,
               777, env={'acc': '[0.03 0.001 0.01]-random', 'gyro': '[6 5 4]d-random'})
    gen_philox('90deg_mid_rf0_vibsin', 'motion_def-90deg_turn.csv', 100.0, 'mid-accuracy', 0, 3,
               778, env={'acc': '[0.03 0.001 0.01]g-3Hz-sinusoidal',
                         'gyro': '[6 5 4]d-0.5Hz-sinusoidal'})
    gen_ned_stats()
    gen_philox_config3()
    gen_philox_white_drift(1)
    gen_philox_white_drift(0)
    gen_philox_psd(1)
    gen_philox_odo(1)
    gen_philox_odo(0)
    gen_gps(0)
    gen_gps(1)
    gen_traj('90deg_turn_100hz_rf1', 'motion_def-90deg_turn.csv', 100.0, 1)
    gen_traj('90deg_turn_100hz_rf0', 'motion_def-90deg_turn.csv', 100.0, 0)
    gen_pathgen()
    gen_allan()
    gen_allan_config4()
    gen_psd()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == '__main__':
    main()
