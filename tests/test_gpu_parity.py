"""GPU parity tests (run on the B200 box): the CUDA path through the C ABI against the
golden vectors produced by the unmodified reference and against the NumPy oracle.
Tolerance: |x - ref| <= 1e-6 * max(|ref|, scale) as BASELINE north_star states (SURVEY 8c);
the observed deviation is ~1e-12 and a tighter bound is asserted beside it."""
import ctypes

import numpy as np
import pytest

import oracle_np as onp
from conftest import allan_golden, load_golden, assert_close, wrap_pi

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')
REL = 1e-6          # the contract
TIGHT = 1e-9        # what the FP64 kernels actually deliver (libm/FMA differences only)
LANES = [1, 2, 4, 8, 16, 32]


@pytest.fixture(scope='module')
def eng():
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from gnss_ins_sim_b200 import engine
    return engine


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def _check_nav(att, pos, vel, g_att, g_pos, g_vel, rel):
    d = wrap_pi(att - g_att)
    assert np.abs(d).max() <= rel, 'att worst %.3e' % np.abs(d).max()
    # rf=1 positions carry a 4.7e6 m ECEF offset: compare displacement too (SURVEY 8c)
    assert_close(pos - pos[..., :1, :], g_pos - g_pos[..., :1, :], rel, 1.0, 'pos-pos0')
    assert_close(pos, g_pos, rel, 1.0, 'pos')
    assert_close(vel, g_vel, rel, 1.0, 'vel')


@pytest.mark.parametrize('lanes', LANES)
@pytest.mark.parametrize('name', ['bosch', 'nxp'])
def test_k2_logged_data(eng, name, lanes):
    g = load_golden('logged_%s.npz' % name)
    ini = _dev(g['ini'][None])
    att, pos, vel = eng.free_integration(0, float(g['fs']), _dev(g['gyro'][None]),
                                         _dev(g['accel'][None]), ini, earth_rot=False,
                                         lanes_per_run=lanes)
    for rel in (REL, TIGHT):
        _check_nav(att.cpu().numpy()[0], pos.cpu().numpy()[0], vel.cpu().numpy()[0],
                   g['att'], g['pos'], g['vel'], rel)


@pytest.mark.parametrize('layout', [0, 1])
@pytest.mark.parametrize('lanes', [0, 1, 4, 32])
@pytest.mark.parametrize('rf', [0, 1])
def test_k2_seeded_reference_noise(eng, rf, lanes, layout):
    g = load_golden('seeded_90deg_rf%d.npz' % rf)
    gyro, accel = g['gyro'], g['accel']
    if layout == 1:
        gyro, accel = gyro.transpose(1, 2, 0), accel.transpose(1, 2, 0)
    att, pos, vel = eng.free_integration(rf, float(g['fs']), _dev(gyro), _dev(accel),
                                         _dev(g['ini'][None]), layout=layout, lanes_per_run=lanes)
    att, pos, vel = [x.cpu().numpy() for x in (att, pos, vel)]
    if layout == 1:
        att, pos, vel = [x.transpose(2, 0, 1) for x in (att, pos, vel)]
    for rel in (REL, TIGHT):
        _check_nav(att, pos, vel, g['att'], g['pos'], g['vel'], rel)


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


PHILOX_TAGS = ['90deg_mid_rf1', '90deg_mid_rf0', '90deg_low_rf1_run1000',
               '90deg_mid_rf1_vibrand', '90deg_mid_rf0_vibsin']


@pytest.mark.parametrize('tag', PHILOX_TAGS)
def test_k1_noise_vs_reference_injection(eng, tag):
    """Device normals == oracle normals; device gyro/accel == reference fed those normals."""
    g = load_golden('philox_%s.npz' % tag)
    ge, ae = _errs(g)
    R, n = g['gyro'].shape[:2]
    run0 = int(g['run_ids'][0])
    gyro, accel, z = eng.imu_noise(float(g['fs']), R, _dev(g['ref_gyro']), _dev(g['ref_accel']),
                                   ge, ae, int(g['seed']), run0, _vib(g, 'vib_gyro'),
                                   _vib(g, 'vib_acc'), dump_z=True)
    zo = onp.noise_normals(n, g['run_ids'], int(g['seed']))
    z = z.cpu().numpy()
    for k, key in enumerate(['acc_gm', 'acc_w', 'gyr_gm', 'gyr_w']):
        assert np.abs(z[:, :, 3 * k:3 * k + 3] - zo[key]).max() < 1e-13, key
    assert_close(gyro.cpu().numpy(), g['gyro'], 1e-12, 1.0, 'gyro')
    assert_close(accel.cpu().numpy(), g['accel'], 1e-12, 1.0, 'accel')
    # TIME_MAJOR layout holds the same numbers
    g2, a2 = eng.imu_noise(float(g['fs']), R, _dev(g['ref_gyro']), _dev(g['ref_accel']), ge, ae,
                           int(g['seed']), run0, _vib(g, 'vib_gyro'), _vib(g, 'vib_acc'),
                           layout=1)
    assert torch.equal(g2.permute(2, 0, 1), gyro) and torch.equal(a2.permute(2, 0, 1), accel)
    # and so does CHANNEL_MAJOR ([R][3][n]: every channel a contiguous series, K4's input)
    g3, a3 = eng.imu_noise(float(g['fs']), R, _dev(g['ref_gyro']), _dev(g['ref_accel']), ge, ae,
                           int(g['seed']), run0, _vib(g, 'vib_gyro'), _vib(g, 'vib_acc'),
                           layout=2)
    assert torch.equal(g3.permute(0, 2, 1), gyro) and torch.equal(a3.permute(0, 2, 1), accel)


def _ref_nav(g):
    return np.concatenate([g['ref_att'], g['ref_pos'], g['ref_vel']], axis=1)


@pytest.mark.parametrize('lanes', LANES)
@pytest.mark.parametrize('tag', PHILOX_TAGS)
def test_k12_fused_mc_vs_reference(eng, tag, lanes):
    """Fused noise+integration+errors == reference pipeline fed the same normals."""
    g = load_golden('philox_%s.npz' % tag)
    ge, ae = _errs(g)
    R, n = g['gyro'].shape[:2]
    rf = int(g['ref_frame'])
    cfg = eng.make_mc_config(rf, float(g['fs']), n, R, int(g['seed']), ge, ae, 1, 9,
                             run_offset=int(g['run_ids'][0]), vib_gyro=_vib(g, 'vib_gyro'),
                             vib_accel=_vib(g, 'vib_acc'), lanes_per_run=lanes, dump_runs=R)
    res = eng.mc_free_integration(cfg, _dev(g['ref_gyro']), _dev(g['ref_accel']),
                                  _dev(_ref_nav(g)), _dev(g['ini'][None]), want_state=True,
                                  dump_nav=True, dump_imu=True)
    att, pos, vel = [x.cpu().numpy() for x in (res.att, res.pos, res.vel)]
    for rel in (REL, 1e-8):
        _check_nav(att, pos, vel, g['att'], g['pos'], g['vel'], rel)
    assert_close(res.gyro.cpu().numpy(), g['gyro'], 1e-12, 1.0, 'gyro')
    assert_close(res.accel.cpu().numpy(), g['accel'], 1e-12, 1.0, 'accel')
    # per-run end-point errors and the end state
    end_state = res.end_state.cpu().numpy()
    assert np.array_equal(end_state[:, 0:3], att[:, -1]) and np.array_equal(end_state[:, 3:6], pos[:, -1])
    err = res.end_err.cpu().numpy()
    g_err = np.concatenate([onp.angle_range_pi(g['att'][:, -1] - g['ref_att'][-1]),
                            g['pos'][:, -1] - g['ref_pos'][-1],
                            g['vel'][:, -1] - g['ref_vel'][-1]], axis=1)
    assert_close(err, g_err, 1e-6, 1e-2, 'end_err')
    # ensemble statistics (K3) against the reference's get_error_stats
    st = eng.error_stats(res.end_err).cpu().numpy()
    for k, key in enumerate(['max', 'avg', 'std']):
        gs = np.concatenate([g['stat_att_euler_' + key], g['stat_pos_' + key], g['stat_vel_' + key]])
        assert_close(st[k], gs, 1e-6, 1e-3, 'stat ' + key)


@pytest.mark.parametrize('lanes', [1, 8, 32])
@pytest.mark.parametrize('rf', [0, 1])
def test_k12_process_error_stats(eng, rf, lanes):
    g = load_golden('philox_90deg_mid_rf%d.npz' % rf)
    ge, ae = _errs(g)
    R, n = g['gyro'].shape[:2]
    start = 250
    cfg = eng.make_mc_config(rf, float(g['fs']), n, R, int(g['seed']), ge, ae, 1, 9,
                             lanes_per_run=lanes, stats_start=start)
    res = eng.mc_free_integration(cfg, _dev(g['ref_gyro']), _dev(g['ref_accel']),
                                  _dev(_ref_nav(g)), _dev(g['ini'][None]))
    ps = res.proc_stats.cpu().numpy()
    for c0, key, ang in ((0, 'att', True), (3, 'pos', False), (6, 'vel', False)):
        o = onp.process_error_stats(g[key], g['ref_' + key], start, ang)
        for k, name in enumerate(['max', 'avg', 'std']):
            assert_close(ps[:, k, c0:c0 + 3], o[name], 1e-6, 1e-4, '%s %s' % (key, name))


def test_k12_sharding_invariance(eng):
    """Runs are keyed by GLOBAL run id: two shards == one launch (multi-GPU contract)."""
    g = load_golden('philox_90deg_mid_rf1.npz')
    ge, ae = _errs(g)
    n = g['ref_gyro'].shape[0]
    args = (_dev(g['ref_gyro']), _dev(g['ref_accel']), _dev(_ref_nav(g)), _dev(g['ini'][None]))
    full = eng.mc_free_integration(eng.make_mc_config(1, 100.0, n, 37, 5, ge, ae, 1, 9,
                                                      lanes_per_run=4), *args).end_err.clone()
    a = eng.mc_free_integration(eng.make_mc_config(1, 100.0, n, 20, 5, ge, ae, 1, 9,
                                                   lanes_per_run=32), *args).end_err.clone()
    b = eng.mc_free_integration(eng.make_mc_config(1, 100.0, n, 17, 5, ge, ae, 1, 9, run_offset=20,
                                                   lanes_per_run=1), *args).end_err.clone()
    assert torch.allclose(torch.cat([a, b]), full, rtol=0, atol=1e-9)
    assert not torch.allclose(a[:17], b, atol=1e-6)      # different runs differ


def test_k2_ini_sets_and_gravity_override(eng):
    """free_integration.py:85-93: run g uses ini set g while g < sets, else set 0;
    row 9 overrides gravity."""
    g = load_golden('seeded_90deg_rf1.npz')
    rng = np.random.RandomState(3)
    S, R = 3, 5
    ini = np.tile(np.append(g['ini'], 9.8)[None], (S, 1))
    ini[:, 3:9] += 1e-3 * rng.randn(S, 6)
    ini[:, 9] = [9.8, 9.79, 9.81]
    gyro = np.tile(g['gyro'][:1], (R, 1, 1))
    accel = np.tile(g['accel'][:1], (R, 1, 1))
    for rf in (0, 1):
        att, pos, vel = eng.free_integration(rf, 100.0, _dev(gyro), _dev(accel), _dev(ini),
                                             lanes_per_run=4)
        sel = np.array([0, 1, 2, 0, 0])
        o_att, o_pos, o_vel = onp.free_integration(rf, 100.0, gyro, accel, ini[sel])
        _check_nav(att.cpu().numpy(), pos.cpu().numpy(), vel.cpu().numpy(), o_att, o_pos, o_vel,
                   TIGHT)


def test_k2_pitch_reflection_and_wrap(eng):
    """Drive pitch through +-pi/2 and yaw/roll through +-pi within a few steps
    (attitude.py:703-720).  The Euler recurrence is singular at pitch = +-pi/2 (1/cos), so
    only a handful of steps are compared: any libm-level difference is amplified by up to
    1/cos^2 per step near the singularity."""
    n, R = 4, 512
    rng = np.random.RandomState(11)
    sign = lambda: rng.choice([-1.0, 1.0], size=R)  # noqa: E731
    ini = np.zeros((R, 9))
    ini[:, 0:3] = [0.55, 2.1, 10.0]
    ini[:, 3:6] = [1.0, 0.2, -0.1]
    ini[:, 6] = sign() * rng.uniform(3.0, 3.14, R)      # yaw near +-pi
    ini[:, 7] = sign() * rng.uniform(1.40, 1.55, R)     # pitch near +-pi/2
    ini[:, 8] = sign() * rng.uniform(3.0, 3.14, R)      # roll near +-pi
    gyro = rng.uniform(-15.0, 15.0, (R, 1, 3)) * np.ones((1, n, 1))
    accel = np.zeros((R, n, 3))
    accel[:, :, 2] = -9.8
    for rf in (0, 1):
        for lanes in (1, 8, 32):
            att, pos, vel = eng.free_integration(rf, 100.0, _dev(gyro), _dev(accel), _dev(ini),
                                                 lanes_per_run=lanes)
            o_att, o_pos, o_vel = onp.free_integration(rf, 100.0, gyro, accel, ini)
            a = att.cpu().numpy()
            # 1/cos(pitch)^2 reaches ~2e3 here: ulp-level differences in sin/cos show up at 1e-8
            assert np.abs(wrap_pi(a - o_att)).max() < 1e-7
            assert_close(vel.cpu().numpy(), o_vel, 1e-7, 1.0, 'vel')
            assert (np.abs(a[:, :, 1]) <= np.pi / 2 + 1e-12).all()
            # yaw / roll get ONE +-2pi wrap per step, not a modulo (attitude.py:712-720): near
            # the singularity a single step can move them by more than 2pi, as in the reference
    # the scenario really exercises the branches
    d_pitch = np.abs(np.diff(o_att[:, :, 1], axis=1))
    flipped = (np.abs(np.abs(np.diff(o_att[:, :, 0], axis=1)) - np.pi) < 0.5).any(1)
    assert flipped.sum() > 20 and d_pitch.max() < 0.2


def test_k3_stats_vs_numpy(eng):
    rng = np.random.RandomState(5)
    for R, nc in ((1, 9), (7, 9), (1000, 9), (100003, 9), (513, 27), (64, 1)):
        e = rng.randn(R, nc) * np.logspace(-6, 3, nc)[None] + np.linspace(-2, 2, nc)[None]
        st = eng.error_stats(_dev(e)).cpu().numpy()
        o = onp.array_stats(e)
        assert_close(st[0], o['max'], 1e-14, 0.0, 'max')
        assert_close(st[1], o['avg'], 1e-9, 1e-9, 'avg')
        assert_close(st[2], o['std'], 1e-11, 0.0, 'std')


def test_k4_allan_vs_reference(eng):
    g = allan_golden()
    x = _dev(g['x'])
    avar, tau = eng.allan(float(g['fs']), x, x.numel(), 1)
    assert_close(tau.cpu().numpy(), g['tau'], 1e-15, 0.0, 'tau')
    assert_close(avar.cpu().numpy()[0], g['avar'], 1e-9, 0.0, 'avar')
    x2 = _dev(g['x2'])
    avar, tau = eng.allan(float(g['fs2']), x2, x2.numel(), 1)
    assert_close(avar.cpu().numpy()[0], g['avar2'], 1e-9, 0.0, 'avar2')
    assert_close(tau.cpu().numpy(), g['tau2'], 1e-15, 0.0, 'tau2')
    a3, t3 = eng.allan(100.0, _dev(g['x3']), 800, 1)       # too short: ([], [])
    assert a3.numel() == 0 and t3.numel() == 0


def test_k4_allan_interleaved_triads(eng):
    """Allan plugin layout: accel/gyro (n,3) per run -> 3 series with sample stride 3."""
    rng = np.random.RandomState(9)
    R, n, fs = 3, 25217, 100.0
    x = rng.randn(R, n, 3) * np.array([1.0, 0.1, 10.0]) + np.array([0.0, 5.0, -9.8])
    x += np.cumsum(1e-3 * rng.randn(R, n, 3), axis=1)
    avar, tau = eng.allan(fs, _dev(x), n, R * 3, inner=3, outer_stride=3 * n, sample_stride=3)
    avar = avar.cpu().numpy().reshape(R, 3, -1)
    for r in range(R):
        for c in range(3):
            o, t = onp.allan_var(x[r, :, c], fs)
            assert_close(avar[r, c], o, 1e-9, 0.0, 'avar %d %d' % (r, c))
    assert_close(tau.cpu().numpy(), t, 1e-15, 0.0, 'tau')


@pytest.mark.parametrize('nser,n', [(1, 5041), (1, 5049), (1, 5050), (1, 10081), (1, 15129), (1, 10090),
                                    (4, 10082), (4, 20170), (3, 5040), (2, 50400)])
def test_k4_allan_ragged_last_chunk(eng, nser, n):
    """The last chunk of a series holds 1 .. 5040 elements: every cluster size must count exactly
    the clusters the reference counts (allan.py:44-57), whatever is left over."""
    rng = np.random.RandomState(n)
    fs = 100.0
    x = 0.7 + rng.randn(nser, n) + np.cumsum(0.01 * rng.randn(nser, n), axis=1)
    avar, tau = eng.allan(fs, _dev(x), n, nser)
    avar = avar.cpu().numpy()
    for r in range(nser):
        o, t = onp.allan_var(x[r], fs)
        assert_close(avar[r], o, 1e-9, 0.0, 'avar %d' % r)
    assert_close(tau.cpu().numpy(), t, 1e-15, 0.0, 'tau')


def test_host_entry_points(eng):
    """The *_host C-ABI calls (host buffers in, host buffers out)."""
    from gnss_ins_sim_b200 import _lib
    lib = _lib.load()
    g = load_golden('philox_90deg_mid_rf1.npz')
    ge, ae = _errs(g)
    R, n = g['gyro'].shape[:2]
    gyro = np.ascontiguousarray(g['gyro'])
    accel = np.ascontiguousarray(g['accel'])
    ini = np.ascontiguousarray(g['ini'][None])
    att, pos, vel = np.empty_like(gyro), np.empty_like(gyro), np.empty_like(gyro)
    hp = _lib.host_ptr
    _lib.check(lib.b2ins_free_integration_f64_host(1, 100.0, R, n, hp(gyro), hp(accel), 0, hp(ini),
                                                   1, 9, 0, 1, hp(att), hp(pos), hp(vel), 0))
    _check_nav(att, pos, vel, g['att'], g['pos'], g['vel'], TIGHT)
    go, ao = np.empty_like(gyro), np.empty_like(gyro)
    se_g, se_a = _lib.sensor_err(ge, 'arw'), _lib.sensor_err(ae, 'vrw')
    rg, ra = np.ascontiguousarray(g['ref_gyro']), np.ascontiguousarray(g['ref_accel'])
    _lib.check(lib.b2ins_imu_noise_f64_host(100.0, R, n, hp(rg), hp(ra), ctypes.byref(se_g),
                                            ctypes.byref(se_a), None, None, int(g['seed']), 0, 0,
                                            hp(go), hp(ao), None))
    assert_close(go, g['gyro'], 1e-12, 1.0, 'gyro')
    cfg = eng.make_mc_config(1, 100.0, n, R, int(g['seed']), ge, ae, 1, 9)
    end_err = np.empty((R, 9))
    stats = np.empty((3, 9))
    nav = np.ascontiguousarray(_ref_nav(g))
    _lib.check(lib.b2ins_mc_free_integration_f64_host(ctypes.byref(cfg), hp(rg), hp(ra), hp(nav),
                                                      hp(ini), hp(end_err), hp(stats)))
    gs = np.concatenate([g['stat_att_euler_std'], g['stat_pos_std'], g['stat_vel_std']])
    assert_close(stats[2], gs, 1e-6, 1e-3, 'std')
    ga = allan_golden()
    x = np.ascontiguousarray(ga['x'])
    avar, tau = np.empty(38), np.empty(38)
    _lib.check(lib.b2ins_allan_f64_host(100.0, x.size, 1, hp(x), 1, x.size, 1, hp(avar), hp(tau)))
    assert_close(avar, ga['avar'], 1e-9, 0.0, 'avar')


def test_argument_errors(eng):
    from gnss_ins_sim_b200 import _lib
    lib = _lib.load()
    x = torch.zeros(4, 10, 3, dtype=torch.float64, device='cuda')
    ini = torch.zeros(1, 9, dtype=torch.float64, device='cuda')
    with pytest.raises(ValueError):
        eng.free_integration(2, 100.0, x, x, ini)                  # bad ref_frame
    with pytest.raises(ValueError):
        eng.free_integration(1, 100.0, x, x, ini, lanes_per_run=3)  # bad lane group
    with pytest.raises(ValueError):
        eng.free_integration(1, 0.0, x, x, ini)
    assert b'' != lib.b2ins_last_error()
    # empty inputs are a no-op
    e = torch.zeros(0, 10, 3, dtype=torch.float64, device='cuda')
    att, pos, vel = eng.free_integration(1, 100.0, e, e, ini)
    assert att.shape == (0, 10, 3)


def test_statistical_sanity_large_ensemble(eng):
    """Size-independent properties at BASELINE config-2 scale (R=1000 and 2^15 runs):
    ensemble means ~ 0 within 5 sigma/sqrt(R); std independent of the lane grouping;
    noise-free run reproduces the trajectory."""
    g = load_golden('traj_90deg_turn_100hz_rf1.npz')
    nav = np.concatenate([g['ref_att'], g['ref_pos'], g['ref_vel']], axis=1)
    n = nav.shape[0]
    mid_g = {'b': np.zeros(3), 'b_drift': np.full(3, 3.5 * np.pi / 180 / 3600),
             'b_corr': np.full(3, 100.0), 'arw': np.full(3, 0.25 * np.pi / 180 / 60)}
    mid_a = {'b': np.zeros(3), 'b_drift': np.full(3, 5e-5), 'b_corr': np.full(3, 100.0),
             'vrw': np.full(3, 0.03 / 60)}
    args = (_dev(g['ref_gyro']), _dev(g['ref_accel']), _dev(nav), _dev(g['ini'][None]))
    stats = {}
    for R, lanes in ((1000, 32), (1000, 1), (32768, 1)):
        cfg = eng.make_mc_config(1, 100.0, n, R, 2024, mid_g, mid_a, 1, 9, lanes_per_run=lanes)
        res = eng.mc_free_integration(cfg, *args)
        stats[(R, lanes)] = eng.error_stats(res.end_err).cpu().numpy()
    a, b, c = stats[(1000, 32)], stats[(1000, 1)], stats[(32768, 1)]
    assert np.abs(a - b).max() < 1e-9                      # same runs, different lane grouping
    assert (np.abs(c[2] / a[2] - 1) < 0.1).all()           # std stable with ensemble size
    # the truth itself has a ~1e-2 m / 1e-4 rad discretisation offset (pathgen vs forward
    # Euler); the noise contribution to the mean shrinks like 1/sqrt(R)
    zero = {k: np.zeros(3) for k in ('b', 'b_drift')}
    quiet_g = dict(zero, b_corr=np.full(3, 100.0), arw=np.zeros(3))
    quiet_a = dict(zero, b_corr=np.full(3, 100.0), vrw=np.zeros(3))
    cfg = eng.make_mc_config(1, 100.0, n, 4, 1, quiet_g, quiet_a, 1, 9, lanes_per_run=2)
    q = eng.mc_free_integration(cfg, *args).end_err.cpu().numpy()
    assert np.abs(q - q[0]).max() == 0.0                   # noise-free runs are identical
    assert (np.abs(c[1] - q[0]) < 5 * c[2] / np.sqrt(32768) + 1e-12).all()


def test_k5_psd_series_vs_oracle(eng):
    """K5 == oracle time_series_from_psd fed the same Philox phase normals (the oracle itself is
    pinned to the reference on tests/golden/psd.npz), for an even n <= 16384 (no tiling, N = n,
    not a power of two), an odd n and n > 16384 (N = 16384), with and without interpolation."""
    g = load_golden('psd.npz')
    freq, sxx = g['freq_a'], g['sxx_a']
    fs = float(g['fs_a'])
    R, seed, run0 = 3, 99, 5
    vib = {'type': 'psd', 'freq': freq, 'x': sxx, 'y': 2.0 * sxx, 'z': 0.5 * sxx + 1e-6}
    for n in (1000, 777, 40001):
        for sensor in (0, 1):
            series, N = eng.psd_series(fs, n, R, sensor, vib, seed, run0)
            assert N == min(n + n % 2, 16384) and tuple(series.shape) == (R, 3, N)
            L = N // 2 + 1
            z = onp.psd_phase_normals(L, np.arange(run0, run0 + R), seed, sensor)
            s = series.cpu().numpy()
            for r in range(R):
                for c, key in enumerate(('x', 'y', 'z')):
                    ok, x = onp.time_series_from_psd(vib[key], freq, fs, n, z[r, c])
                    assert ok
                    assert_close(np.resize(s[r, c], n) if n > N else s[r, c][:n], x, 1e-9,
                                 np.abs(x).max(), 'psd series n=%d' % n)
    # a table that already has L rows is used as it is (no interpolation)
    n = 1000
    L = n // 2 + 1
    f2 = np.linspace(0, fs / 2, L)
    vib2 = {'type': 'psd', 'freq': f2, 'x': np.interp(f2, freq, sxx), 'y': np.ones(L), 'z': np.zeros(L) + 1e-3}
    series, N = eng.psd_series(fs, n, 1, 0, vib2, 1, 0)
    z = onp.psd_phase_normals(L, [0], 1, 0)
    ok, x = onp.time_series_from_psd(vib2['x'], f2, fs, n, z[0, 0])
    assert_close(series.cpu().numpy()[0, 0], x, 1e-9, np.abs(x).max(), 'no-interp')


def test_k5_psd_vibration_through_the_fused_kernel(eng):
    """PSD vibration inside K12/K1: gyro/accel histories == oracle noise + oracle PSD series."""
    g = load_golden('philox_90deg_mid_rf1.npz')
    p = load_golden('psd.npz')
    ge, ae = _errs(g)
    n = g['ref_gyro'].shape[0]
    R, seed = 2, 31
    from gnss_ins_sim_b200.sim import parse_env
    vib = parse_env(np.column_stack([p['freq_a'], p['sxx_a'], p['sxx_a'] * 0.3, p['sxx_a'] * 2]), 100.0)
    assert vib['type'] == 'psd' and vib['freq'][-1] <= 50.0
    sa, N = eng.psd_series(100.0, n, R, 0, vib, seed, 0)
    sg, _ = eng.psd_series(100.0, n, R, 1, vib, seed, 0)
    gyro, accel = eng.imu_noise(100.0, R, _dev(g['ref_gyro']), _dev(g['ref_accel']), ge, ae, seed, 0,
                                eng.vib_series(sg, N), eng.vib_series(sa, N))
    L = N // 2 + 1
    o_gyro, o_accel = onp.imu_noise(100.0, g['ref_gyro'], g['ref_accel'], ge, ae, seed, np.arange(R))
    for sensor, dev_out, base in ((0, accel, o_accel), (1, gyro, o_gyro)):
        z = onp.psd_phase_normals(L, np.arange(R), seed, sensor)
        for r in range(R):
            for c, key in enumerate(('x', 'y', 'z')):
                ok, x = onp.time_series_from_psd(vib[key], vib['freq'], 100.0, n, z[r, c])
                assert_close(dev_out.cpu().numpy()[r, :, c], base[r, :, c] + x, 1e-9, 1.0, 'meas+psd')
