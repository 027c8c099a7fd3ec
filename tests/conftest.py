import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'oracle'))
GOLDEN = os.path.join(ROOT, 'tests', 'golden')


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box)')


def load_golden(name):
    return dict(np.load(os.path.join(GOLDEN, name), allow_pickle=False))


def allan_golden():
    """allan.npz with its 180 000-sample series `x` regenerated from the stored seed, as
    oracle/gen_golden.py made it (NumPy's RandomState stream is frozen); every 1000th stored
    sample pins the regeneration."""
    g = load_golden('allan.npz')
    n = int(g['n'])
    rng = np.random.RandomState(int(g['seed']))
    g['x'] = 0.01 * rng.randn(n) + np.cumsum(1e-5 * rng.randn(n))
    assert np.array_equal(g['x'][::1000], g['x_every_1000']), 'allan.npz: regenerated series differs'
    return g


@pytest.fixture(scope='session')
def golden():
    return load_golden


def assert_close(x, ref, rel=1e-6, scale=1.0, what=''):
    """|x - ref| <= rel * max(|ref|, scale)  (SURVEY 8c tolerance note)."""
    x = np.asarray(x, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    assert x.shape == ref.shape, (what, x.shape, ref.shape)
    tol = rel * np.maximum(np.abs(ref), scale)
    bad = np.abs(x - ref) > tol
    assert not bad.any(), '%s: %d/%d out of tolerance, worst |d|=%.3e (tol %.3e)' % (
        what, bad.sum(), bad.size, np.abs(x - ref).max(), tol.min())


def wrap_pi(x):
    return (np.asarray(x) + np.pi) % (2 * np.pi) - np.pi


def write_logged_dir(path, g, deg=True):
    """A logged-data directory in the reference's file format (demo_data_files/*): time.csv,
    gyro-0.csv in deg/s, accel-0.csv, all-zero reference files, from a golden 'logged' fixture."""
    os.makedirs(path, exist_ok=True)
    n = g['gyro'].shape[0]
    r2d = 180.0 / np.pi if deg else 1.0
    gu = 'deg/s' if deg else 'rad/s'
    np.savetxt(os.path.join(path, 'time.csv'), np.arange(n) / float(g['fs']), header='time (sec)', comments='')
    np.savetxt(os.path.join(path, 'gyro-0.csv'), g['gyro'] * r2d, delimiter=',', comments='',
               header='gyro_x (%s),gyro_y (%s),gyro_z (%s)' % (gu, gu, gu), fmt='%.18e')
    np.savetxt(os.path.join(path, 'accel-0.csv'), g['accel'], delimiter=',', comments='',
               header='accel_x (m/s^2),accel_y (m/s^2),accel_z (m/s^2)', fmt='%.18e')
    z = np.zeros((n, 3))
    np.savetxt(os.path.join(path, 'ref_pos.csv'), z, delimiter=',', comments='',
               header='ref_pos_lat (deg),ref_pos_lon (deg),ref_pos_alt (m)')
    np.savetxt(os.path.join(path, 'ref_vel.csv'), z, delimiter=',', comments='',
               header='ref_vel_x (m/s),ref_vel_y (m/s),ref_vel_z (m/s)')
    np.savetxt(os.path.join(path, 'ref_att_euler.csv'), z, delimiter=',', comments='',
               header='ref_Yaw (deg),ref_Pitch (deg),ref_Roll (deg)')
    with open(os.path.join(path, 'notes.txt'), 'w') as f:
        f.write('not a data file')
    return path
