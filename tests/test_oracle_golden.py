"""Pin the NumPy oracle (oracle/oracle_np.py) against vectors produced by the
unmodified reference (oracle/gen_golden.py).  CPU only."""
import numpy as np
import pytest

import oracle_np as onp
from conftest import allan_golden, load_golden, assert_close, wrap_pi

TIGHT = 1e-12


@pytest.mark.parametrize('name', ['bosch', 'nxp'])
def test_logged_data_rf0(name):
    g = load_golden('logged_%s.npz' % name)
    att, pos, vel = onp.free_integration(0, float(g['fs']), g['gyro'][None], g['accel'][None],
                                         g['ini'][None], earth_rot=False)
    assert_close(att[0], g['att'], TIGHT, what='att')
    assert_close(pos[0], g['pos'], TIGHT, what='pos')
    assert_close(vel[0], g['vel'], TIGHT, what='vel')


@pytest.mark.parametrize('rf', [0, 1])
def test_seeded_reference_noise(rf):
    g = load_golden('seeded_90deg_rf%d.npz' % rf)
    ini = np.tile(g['ini'], (2, 1))
    att, pos, vel = onp.free_integration(rf, float(g['fs']), g['gyro'], g['accel'], ini)
    assert_close(att, g['att'], TIGHT, what='att')
    assert_close(pos - pos[:, :1], g['pos'] - g['pos'][:, :1], TIGHT, what='pos-pos0')
    assert_close(pos, g['pos'], TIGHT, what='pos')
    assert_close(vel, g['vel'], TIGHT, what='vel')


def _errs(g):
    return ({'b': g['gyro_b'], 'b_drift': g['gyro_b_drift'], 'b_corr': g['gyro_b_corr'],
             'arw': g['gyro_arw']},
            {'b': g['accel_b'], 'b_drift': g['accel_b_drift'], 'b_corr': g['accel_b_corr'],
             'vrw': g['accel_vrw']})


def _vib(g, key):
    if key + '_type' not in g:
        return None
    a = g[key + '_amp']
    return {'type': str(g[key + '_type']), 'x': a[0], 'y': a[1], 'z': a[2],
            'freq': float(g[key + '_freq'])}


@pytest.mark.parametrize('tag', ['90deg_mid_rf1', '90deg_mid_rf0', '90deg_low_rf1_run1000',
                                 '90deg_mid_rf1_vibrand', '90deg_mid_rf0_vibsin'])
def test_philox_stream_through_reference(tag):
    """oracle noise + mechanization + stats == reference fed the same normals."""
    g = load_golden('philox_%s.npz' % tag)
    ge, ae = _errs(g)
    fs, rf = float(g['fs']), int(g['ref_frame'])
    gyro, accel = onp.imu_noise(fs, g['ref_gyro'], g['ref_accel'], ge, ae, int(g['seed']),
                                g['run_ids'], _vib(g, 'vib_acc'), _vib(g, 'vib_gyro'))
    assert_close(gyro, g['gyro'], TIGHT, what='gyro')
    assert_close(accel, g['accel'], TIGHT, what='accel')
    R = gyro.shape[0]
    att, pos, vel = onp.free_integration(rf, fs, gyro, accel, np.tile(g['ini'], (R, 1)))
    assert_close(att, g['att'], 1e-10, what='att')
    assert_close(pos, g['pos'], 1e-10, what='pos')
    assert_close(vel, g['vel'], 1e-10, what='vel')
    st = onp.end_point_error_stats(att, pos, vel, g['ref_att'], g['ref_pos'], g['ref_vel'])
    for name in ('att_euler', 'pos', 'vel'):
        for k in ('max', 'avg', 'std'):
            assert_close(st[name][k], g['stat_%s_%s' % (name, k)], 1e-7, 1e-3,
                         what='%s %s' % (name, k))


def test_philox_known_answer():
    """Philox4x32-10 KAT from the Random123 distribution (kat_vectors):
    ctr=0,key=0 ; ctr=ff..,key=ff.. ; ctr=pi digits,key=e digits... (first two)."""
    x = onp.philox4x32_10(0, 0, 0, 0, 0, 0)
    assert [int(v) for v in x] == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    f = 0xFFFFFFFF
    x = onp.philox4x32_10(f, f, f, f, f, f)
    assert [int(v) for v in x] == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    x = onp.philox4x32_10(0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344, 0xa4093822, 0x299f31d0)
    assert [int(v) for v in x] == [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_normals_are_standard():
    z0, z1 = onp.normal_pair(np.arange(200000), 0, 5, 42)
    z = np.concatenate([z0, z1])
    assert abs(z.mean()) < 0.01 and abs(z.std() - 1) < 0.01
    assert abs(np.mean(z ** 3)) < 0.03 and abs(np.mean(z ** 4) - 3) < 0.06
    assert abs(np.corrcoef(z0, z1)[0, 1]) < 0.01
    assert np.isfinite(z).all()


def test_allan_matches_reference():
    g = allan_golden()
    avar, tau = onp.allan_var(g['x'], float(g['fs']))
    assert_close(tau, g['tau'], 1e-15, what='tau')
    assert_close(avar, g['avar'], 1e-12, 0.0, what='avar')
    assert len(tau) == 38
    avar, tau = onp.allan_var(g['x2'], float(g['fs2']))
    assert_close(avar, g['avar2'], 1e-12, 0.0, what='avar2')
    assert_close(tau, g['tau2'], 1e-15, what='tau2')
    a, t = onp.allan_var(g['x3'], 100.0)
    assert len(a) == 0 and len(t) == 0


@pytest.mark.parametrize('tag', ['a', 'b'])
def test_psd_matches_reference(tag):
    g = load_golden('psd.npz')
    ok, x = onp.time_series_from_psd(g['sxx_' + tag], g['freq_' + tag], float(g['fs_' + tag]),
                                     int(g['n_' + tag]), g['z_' + tag])
    assert ok
    assert_close(x, g['x_' + tag], 1e-12, what='psd series')


def test_golden_survey_values():
    """The end values quoted in SURVEY 8(c) are the ones in the fixtures."""
    g = load_golden('logged_bosch.npz')
    assert_close(g['att'][-1], [-0.04581388717726487, -0.01158326991382768, -0.0113185715399397],
                 1e-14)
    g = load_golden('seeded_90deg_rf1.npz')
    assert_close(g['att'][0, -1], [7.8534050869474481e-01, -2.0678960287434905e-04,
                                   9.5098666116010674e-05], 1e-13)
    assert_close(g['pos'][0, -1], [-2707376.9803619734, 4688713.859123157, 3360102.3087808033],
                 1e-15)


@pytest.mark.parametrize('rf', [0, 1])
def test_odometer_variant_oracle(rf):
    """odo_gen + free_integration_odo restatements == reference fed the same normals."""
    g = load_golden('philox_90deg_mid_rf%d_odo.npz' % rf)
    R, n = g['odo'].shape
    zo = onp.odo_normals(n, g['run_ids'], int(g['seed']))
    odo = onp.odo_gen(g['ref_odo'], {'scale': float(g['odo_scale']), 'stdv': float(g['odo_stdv'])}, zo)
    assert_close(odo, g['odo'], TIGHT, what='odo')
    att, pos, vel = onp.free_integration_odo(rf, 100.0, g['gyro'], odo, np.tile(g['ini'], (R, 1)))
    assert_close(att, g['att'], 1e-10, what='att')
    assert_close(pos, g['pos'], 1e-10, what='pos')
    assert_close(vel, g['vel'], 1e-10, what='vel')


@pytest.mark.parametrize('rf', [0, 1])
def test_gps_gen_oracle(rf):
    """gps_gen restatement == pathgen.gps_gen (pathgen.py:596-625) fed the same normals."""
    g = load_golden('gps_90deg_rf%d.npz' % rf)
    R, m, _ = g['gps'].shape
    z = onp.gps_normals(m, g['run_ids'], int(g['seed']))
    out = onp.gps_gen(g['ref_gps'], {'stdp': g['stdp'], 'stdv': g['stdv']}, rf, z)
    assert np.array_equal(out, g['gps'])
    # the metre -> radian conversion really happened (LLA) / did not (xyz)
    sd = (out - g['ref_gps'][None]).std(axis=(0, 1))
    assert (sd[0] < 1e-5) == (rf == 0) and abs(sd[2] / 7.0 - 1) < 0.2 and abs(sd[4] / 0.05 - 1) < 0.2


def _errs(g):
    ge = {'b': g['gyro_b'], 'b_drift': g['gyro_b_drift'], 'b_corr': g['gyro_b_corr'], 'arw': g['gyro_arw']}
    ae = {'b': g['accel_b'], 'b_drift': g['accel_b_drift'], 'b_corr': g['accel_b_corr'], 'vrw': g['accel_vrw']}
    return ge, ae


@pytest.mark.parametrize('rf', [0, 1])
def test_white_bias_drift_branch_is_pinned(rf):
    """b_corr = inf (a dict IMU without *_b_corr): drift[i]*randn(n), pathgen.py:591-593 -- both oracles
    against the reference fed the same normals (philox_90deg_whitedrift_rf*.npz)."""
    import oracle_c
    g = load_golden('philox_90deg_whitedrift_rf%d.npz' % rf)
    ge, ae = _errs(g)
    assert np.all(np.isinf(ge['b_corr'])) and np.all(np.isinf(ae['b_corr']))
    R = g['gyro'].shape[0]
    for mod in (onp, oracle_c):
        gyro, accel = mod.imu_noise(100.0, g['ref_gyro'], g['ref_accel'], ge, ae, int(g['seed']), g['run_ids'])
        assert_close(gyro, g['gyro'], TIGHT, what='gyro')
        assert_close(accel, g['accel'], TIGHT, what='accel')
    att, pos, vel = onp.free_integration(rf, 100.0, g['gyro'], g['accel'], np.tile(g['ini'], (R, 1)))
    assert_close(att, g['att'], 1e-10, what='att')
    assert_close(vel, g['vel'], 1e-10, what='vel')


def test_psd_vibration_through_the_reference_sim_is_pinned():
    """env = PSD tables: the oracle's time_series_from_psd on the b2ins phase normals, added by
    sensor_gen, equals what the reference Sim produced (philox_90deg_mid_rf1_psd.npz)."""
    g = load_golden('philox_90deg_mid_rf1_psd.npz')
    n, fs, seed = 1000, 100.0, int(g['seed'])
    L = n // 2 + 1
    z = onp.noise_normals(n, g['run_ids'], seed)
    imu_g = {'b': np.zeros(3), 'b_drift': np.full(3, 3.5 * np.pi / 180 / 3600), 'b_corr': np.full(3, 100.0),
             'arw': np.full(3, 0.25 * np.pi / 180 / 60)}
    imu_a = {'b': np.zeros(3), 'b_drift': np.full(3, 5e-5), 'b_corr': np.full(3, 100.0), 'vrw': np.full(3, 0.03 / 60)}
    for sensor, tab, ref, err, key, zg, zw, out in (
            (0, g['env_acc'], g['ref_accel'], imu_a, 'vrw', z['acc_gm'], z['acc_w'], g['accel']),
            (1, g['env_gyro'], g['ref_gyro'], imu_g, 'arw', z['gyr_gm'], z['gyr_w'], g['gyro'])):
        m = np.where(tab[:, 0] > 0.5 * fs)[0][0]        # Sim.__parse_env cuts the table at fs/2
        zp = onp.psd_phase_normals(L, g['run_ids'], seed, sensor)
        for r in range(len(g['run_ids'])):
            vib = np.stack([onp.time_series_from_psd(tab[:m, 1 + c], tab[:m, 0], fs, n, zp[r, c])[1]
                            for c in range(3)], axis=1)
            mea = onp.sensor_gen(fs, ref, err, key, zg[r:r + 1], zw[r:r + 1], vib=vib[None])[0]
            assert_close(mea, out[r], 1e-11, what='sensor %d run %d' % (sensor, r))


def test_config3_full_length_oracle_against_the_reference():
    """BASELINE config 3 at its full length (193 036 samples @200 Hz, 'low-accuracy', ref_frame 0): the
    C oracle on the host path generator's trajectory against the end points the unmodified reference
    reached on its own trajectory with the same injected normals (philox_config3_long_drive_rf0.npz)."""
    import os
    import oracle_c
    from conftest import ROOT
    from gnss_ins_sim_b200 import imu_model
    from gnss_ins_sim_b200.sim import trajectory_from_motion_def
    g = load_golden('philox_config3_long_drive_rf0.npz')
    csv = os.path.join(ROOT, 'tests', 'golden', 'motion_def-long_drive.csv')
    t = trajectory_from_motion_def(float(g['fs']), csv, 0)
    n = int(g['n'])
    assert t['ref_gyro'].shape == (n, 3)
    nav_end = np.concatenate([t['ref_att'][-1], t['ref_pos'][-1], t['ref_vel'][-1]])
    # the two trajectories agree row by row (tests/test_cpu_host.py); their last rows here
    assert np.abs(wrap_pi(nav_end[0:3] - g['ref_end'][0:3])).max() < 1e-11
    assert np.abs(nav_end[3:5] - g['ref_end'][3:5]).max() < 1e-13 and abs(nav_end[5] - g['ref_end'][5]) < 1e-6
    imu = imu_model.IMU(accuracy='low-accuracy', axis=6, gps=False)
    R = len(g['run_ids'])
    err, _ = oracle_c.mc_free_integration(0, float(g['fs']), R, int(g['run_ids'][0]), t['ref_gyro'], t['ref_accel'],
                                          nav_end, imu.gyro_err, imu.accel_err, int(g['seed']), g['ini'][None],
                                          threads=0)
    want = g['end_state'] - g['ref_end'][None]
    want[:, 0:3] = wrap_pi(want[:, 0:3])
    # the contract is 1e-6 relative; after 1.9e5 steps the end points are ~1e3 m / 30 m/s off the truth
    assert np.abs(wrap_pi(err[:, 0:3] - want[:, 0:3])).max() < 1e-9
    assert np.abs(err[:, 6:9] - want[:, 6:9]).max() < 1e-6
    assert np.abs((err[:, 3:5] - want[:, 3:5]) * 6.4e6).max() < 1e-4 and np.abs(err[:, 5] - want[:, 5]).max() < 1e-4


def test_config4_full_length_allan_oracle_against_the_reference():
    """BASELINE config 4 at its full length (14.4 M samples @400 Hz): the C oracle's allan_var against
    allan.allan_var of the unmodified reference on the same series (allan_config4_full_length.npz)."""
    import oracle_c
    from gnss_ins_sim_b200 import imu_model
    g = load_golden('allan_config4_full_length.npz')
    n, fs = int(g['n']), float(g['fs'])
    imu = imu_model.IMU(accuracy='low-accuracy', axis=6, gps=False)
    ref_gyro = np.zeros((n, 3))
    ref_accel = np.tile(np.array([4.9, 0.0, -8.487]), (n, 1))
    og, oa = oracle_c.imu_noise(fs, ref_gyro, ref_accel, imu.gyro_err, imu.accel_err, int(g['seed']), [int(g['run'])])
    av, tau = oracle_c.allan_var(np.ascontiguousarray(og[0, :, 2]), fs)
    assert_close(tau, g['tau'], 1e-12, 0.0, 'tau')
    assert_close(av, g['avar_gyro_z'], 1e-10, 0.0, 'avar gyro z')
    av, _ = oracle_c.allan_var(np.ascontiguousarray(oa[0, :, 0]), fs)
    # (a 4.9 m/s^2 offset under increments of 1e-4: the bin means cancel to ~1e-17 absolute either way)
    assert_close(av, g['avar_accel_x'], 1e-7, 0.0, 'avar accel x')
