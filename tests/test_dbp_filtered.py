"""Filtered digital backpropagation (pmx_dbp_set_filter, DbpPlan.set_filter, dbp_plan / pmx.dbp filter_bw,
tests/dbp_oracle.py with bw=): a Gaussian low-pass on the intensity of every backward nonlinear step."""
import ctypes
import math

import numpy as np
import pytest

import oracle.fiber_oracle as orc
import dbp_oracle
import polmux_b200 as pmx
from polmux_b200 import _lib, mc
from polmux_b200.dbp import dbp_plan
from polmux_b200.fiber import fiber_setup
from common import _cols, _mc_scenario, base_fiber, make_tx, rel_l2, scalar_tx

GAIN_DB = 16.0
G16 = 10 ** (GAIN_DB / 10)


def _setup(nsymb, nt, nch=1, pavg_mw=4.0, manakov=False, flag='g-s-', length=8e4):
    gs = make_tx(nsymb, nt, nch=nch, ftype='sepfields' if nch > 1 else 'unique', pavg_mw=pavg_mw)
    s = fiber_setup(base_fiber(length=length, slope=0.057, dphimax=0.02), flag)
    s.manakov = manakov
    return gs, s


def _man(s):
    return 'yes' if s.manakov else 'no'


def _forward(ux, uy, s, nspan, gain):
    for _ in range(nspan):
        _, _, ux, uy, _, _ = orc.matrix_ssfm(ux, uy, s.betat, s.db1, s.dzmaxt, s.dphimaxt, s.gam, s.alphalin, s.nfc,
                                             s.length, 1, _man(s), s.fls, s.brf)
        if gain is not None:
            ux, uy = ux * math.sqrt(gain), uy * math.sqrt(gain)
    return ux, uy


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_oracle_without_filter_is_the_existing_oracles():
    gs, s = _setup(64, 16, nch=3, manakov=False)
    kw = dict(nspan=2, gain=G16, steps_per_span=3)
    a = dbp_oracle.dbp(gs.FIELDX, gs.FIELDY, s.betat, s.gam, s.alphalin, s.nfc, s.length, 'no', bw=None, **kw)
    b = dbp_oracle.dbp(gs.FIELDX, gs.FIELDY, s.betat, s.gam, s.alphalin, s.nfc, s.length, 'no', **kw)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    u = scalar_tx(32, 32, 3, pavg=8.0).FIELDX
    ss = fiber_setup(base_fiber(length=1e5, slope=0.057), 'g-sx')
    a = dbp_oracle.dbp_scalar(u, ss.betat, ss.gam, ss.alphalin, ss.nfc, ss.length, 1, 1, bw=None, **kw)
    b = dbp_oracle.dbp_scalar(u, ss.betat, ss.gam, ss.alphalin, ss.nfc, ss.length, 1, 1, **kw)
    assert np.array_equal(a, b)


@pytest.mark.parametrize('manakov', [False, True])
def test_oracle_wide_filter_is_unfiltered_and_xi0_ignores_the_filter(manakov):
    gs, s = _setup(16, 16, nch=2, pavg_mw=10.0, manakov=manakov)   # 2^8: 1 - H(N/2) = 5.7e-13 at bw = 1e8 bins
    args = (gs.FIELDX, gs.FIELDY, s.betat, s.gam, s.alphalin, s.nfc, s.length, _man(s))
    kw = dict(nspan=2, gain=G16, steps_per_span=2)
    ref = dbp_oracle.dbp(*args, **kw)
    wide = dbp_oracle.dbp(*args, bw=1e8, **kw)
    assert rel_l2(*wide, *ref) <= 1e-12
    lin = [dbp_oracle.dbp(*args, xi=0.0, bw=bw, **kw) for bw in (None, 3.0, 40.0)]
    assert rel_l2(*lin[1], *lin[0]) <= 1e-15 and rel_l2(*lin[2], *lin[0]) <= 1e-15
    u = scalar_tx(32, 32, 3, pavg=8.0).FIELDX
    ss = fiber_setup(base_fiber(length=1e5, slope=0.057), 'g-sx')
    sa = (u, ss.betat, ss.gam, ss.alphalin, ss.nfc, ss.length, 1, 1)
    r = dbp_oracle.dbp_scalar(*sa, **kw)
    w = dbp_oracle.dbp_scalar(*sa, bw=1e9, **kw)   # 2^10: 1 - H(N/2) = 9e-14
    assert np.linalg.norm(w - r) <= 1e-12 * np.linalg.norm(r)


@pytest.mark.parametrize('manakov', [False, True])
def test_filtered_nonlinear_step_keeps_every_modulus(manakov):
    gs, s = _setup(64, 16, pavg_mw=30.0, manakov=manakov)
    ux, uy = gs.FIELDX.copy(), gs.FIELDY.copy()
    op = dbp_oracle.intensity(ux.shape[0], bw=5.0)
    vx, vy = dbp_oracle.matrix_nl_step(manakov, s.alphalin, -np.asarray(s.gam), s.length, ux.copy(), uy.copy(), 1, 1, op)
    p0 = np.abs(ux) ** 2 + np.abs(uy) ** 2
    p1 = np.abs(vx) ** 2 + np.abs(vy) ** 2
    assert np.max(np.abs(p1 - p0) / np.maximum(p0, 1e-300)) <= 1e-13
    if manakov:   # a common phase: each polarization keeps its own modulus
        assert np.max(np.abs(np.abs(vx) - np.abs(ux))) <= 1e-13 * np.max(np.abs(ux))
    u = scalar_tx(32, 32, 3, pavg=8.0).FIELDX
    w = dbp_oracle.nl_step(0.0, -1.3 * np.ones((1, 3)), 1e5, u, 3, 1, 1, dbp_oracle.intensity(u.shape[0], bw=4.0))
    assert np.max(np.abs(np.abs(w) - np.abs(u))) <= 1e-13 * np.max(np.abs(u))


def test_filtered_dbp_beats_plain_dbp_at_one_step_per_span():
    """one 28 Gbaud channel, two polarizations, 3 x 80 km, strongly nonlinear, noise-free; forward at the oracle's own fine
    steps: at one step per span the best filtered residual over a (bw, xi) grid is below the best unfiltered one"""
    nsymb, nt = 512, 8
    gs, s = _setup(nsymb, nt, pavg_mw=8.0, manakov=True)
    s.dphimaxt = 0.005
    ux, uy = _forward(gs.FIELDX.copy(), gs.FIELDY.copy(), s, 3, G16)
    args = (ux, uy, s.betat, s.gam, s.alphalin, s.nfc, s.length, _man(s))
    xis = (0.5, 0.6, 0.7, 0.8, 0.9, 1.0)
    bws_ghz = (2.0, 4.0, 8.0, 16.0)

    def res(**kw):
        return rel_l2(*dbp_oracle.dbp(*args, nspan=3, gain=G16, **kw), gs.FIELDX, gs.FIELDY)
    plain = min(res(steps_per_span=1, xi=xi) for xi in xis)
    filt = min((res(steps_per_span=1, xi=xi, bw=b * nsymb / 28.0), b, xi) for b in bws_ghz for xi in xis)
    four = min(res(steps_per_span=4, xi=xi) for xi in xis)
    lin = res(steps_per_span=1, xi=0.0)
    print('filtered DBP, 3 x 80 km, 1 step/span: linear %.4e, plain %.4e, filtered %.4e (bw %g GHz, xi %g), '
          'plain at 4 steps/span %.4e' % (lin, plain, filt[0], filt[1], filt[2], four))
    assert filt[0] < plain < lin


def test_set_filter_rejects_invalid_bandwidths():
    lib = _lib.load()
    for bw in (-1.0, float('nan'), float('inf')):
        assert lib.pmx_dbp_set_filter(None, bw) == _lib.PMX_ERR_INVALID
    assert lib.pmx_dbp_set_filter(None, 1.0) == _lib.PMX_ERR_INVALID


def test_native_mc_rejects_filter_bw():
    s = fiber_setup(base_fiber(), 'g-s-')
    with pytest.raises(ValueError, match='filter_bw'):
        mc.run_mc_native(s, None, None, None, 16, 16, 1, 16.0, 5.0, 1, 1, receiver={}, dbp_params=dict(filter_bw=10.0))


# ---------------------------------------------------------------------------------------------------------------- GPU
def _run(ctx, s, xs, ys, bw, precision='f64', launches=None, plates=None, **kw):
    b = xs.shape[0]
    fld = _lib.DeviceField(ctx, s.nfft, s.nfc, b, precision={'f64': _lib.PMX_F64, 'f32': _lib.PMX_F32}[precision])
    fld.upload(xs, ys)
    plan = dbp_plan(ctx, s, batch=b, precision=precision, plates=plates, **kw)
    if bw:
        plan.set_filter(bw)
    n0 = ctx.launches
    plan.execute(fld)
    if launches is not None:
        assert ctx.launches - n0 == launches
    plan.close()
    out = fld.download()
    fld.close()
    return out


TWO_POL = [  # nsymb, nt, nch, manakov, nspan, batch, bw (bins)
    (16, 16, 1, False, 2, 1, 6.0),        # 2^8, on-chip
    (64, 16, 1, True, 2, 2, 10.0),        # 2^10
    (128, 16, 3, False, 1, 1, 20.0),      # 2^11, three columns
    (256, 16, 1, False, 2, 1, 30.0),      # 2^12, three passes
    (1024, 16, 1, True, 1, 3, 100.0),     # 2^14, odd batch*nfc
    (4096, 16, 1, False, 2, 1, 300.0),    # 2^16
    (4096, 16, 1, True, 1, 2, 300.0),
]


@pytest.mark.gpu
@pytest.mark.parametrize('case', TWO_POL, ids=lambda c: '%dx%d-nfc%d-%s-%dspan-b%d-bw%g' % (c[0], c[1], c[2], 'man' if c[3] else 'cnlse', c[4], c[5], c[6]))
def test_two_pol_filtered_dbp_matches_the_oracle(ctx, case):
    nsymb, nt, nch, manakov, nspan, batch, bw = case
    gs, s = _setup(nsymb, nt, nch=nch, pavg_mw=10.0, manakov=manakov)
    g = G16 if nspan > 1 else None
    kw = dict(nspan=nspan, steps_per_span=3)
    xs = np.concatenate([_cols(np.roll(gs.FIELDX, 7 * b, axis=0)) for b in range(batch)])
    ys = np.concatenate([_cols(np.roll(gs.FIELDY, -5 * b, axis=0)) for b in range(batch)])
    onchip = s.nfft < 4096
    gx, gy = _run(ctx, s, xs, ys, bw, launches=1 if onchip else None, gain_db=GAIN_DB if g else None, **kw)
    errs = []
    for b in range(batch):
        wx, wy = dbp_oracle.dbp(xs[b].T, ys[b].T, s.betat, s.gam, s.alphalin, s.nfc, s.length, _man(s), gain=g, bw=bw,
                                **kw)
        errs.append(rel_l2(gx[b].T, gy[b].T, wx, wy))
        if b == 0:   # the filter changes the result
            ux, uy = dbp_oracle.dbp(xs[b].T, ys[b].T, s.betat, s.gam, s.alphalin, s.nfc, s.length, _man(s), gain=g, **kw)
            assert rel_l2(wx, wy, ux, uy) > 1e-6
    print('filtered dbp parity %s: rel_l2 %s' % (case, ['%.3e' % e for e in errs]))
    assert max(errs) <= 1e-10, errs


@pytest.mark.gpu
@pytest.mark.parametrize('nsymb', [64, 1024])
def test_pmd_filtered_dbp_matches_the_oracle(ctx, nsymb):
    """PMD-aware, per-realization plates: on-chip (2^10) and three passes (2^14)"""
    gs = make_tx(nsymb, 16, pavg_mw=10.0)
    fib = base_fiber(length=8e4, slope=0.057, dphimax=0.02, dgd=0.5, nplates=12, manakov='no')
    s = fiber_setup(fib, 'gps-', rng=np.random.Generator(np.random.PCG64(7)))
    nspan, batch, bw = 2, 2, nsymb / 8.0
    # [realization][span] plate draws
    brfs = [[dict(zip(('db0', 'theta', 'epsilon'), mc.draw_plates(mc.plate_seed(b, k), s.nplates))) for k in range(nspan)]
            for b in range(batch)]
    plates = tuple(np.array([[brfs[b][k][n] for b in range(batch)] for k in range(nspan)])
                   for n in ('db0', 'theta', 'epsilon'))
    xs = np.concatenate([_cols(np.roll(gs.FIELDX, 9 * b, axis=0)) for b in range(batch)])
    ys = np.concatenate([_cols(gs.FIELDY) for b in range(batch)])
    kw = dict(nspan=nspan, steps_per_span=2)
    gx, gy = _run(ctx, s, xs, ys, bw, plates=plates, gain_db=GAIN_DB, **kw)
    db1 = np.asarray(s.db1)
    for b in range(batch):
        wx, wy = dbp_oracle.dbp_pmd(xs[b].T, ys[b].T, s.betat, db1, s.gam, s.alphalin, 1, s.length, _man(s), brfs[b],
                                    gain=G16, bw=bw, **kw)
        err = rel_l2(gx[b].T, gy[b].T, wx, wy)
        print('filtered pmd dbp 2^%d b%d: %.3e' % (int(np.log2(s.nfft)), b, err))
        assert err <= 1e-10


SCALAR = [  # nsymb, nt, nch, flag, bw
    (32, 32, 1, 'g-sx', 8.0),     # ex06_ber.m
    (64, 32, 5, 'g-sx', 16.0),    # ex10_wdm.m
    (128, 32, 1, 'g-s-', 30.0),   # 2^12
]


@pytest.mark.gpu
@pytest.mark.parametrize('case', SCALAR, ids=lambda c: '%dx%dx%d-%s-bw%g' % c)
def test_scalar_filtered_dbp_matches_the_oracle(ctx, case):
    nsymb, nt, nch, flag, bw = case
    scalar_tx(nsymb, nt, nch, pavg=8.0)
    s = fiber_setup(base_fiber(length=1e5, dphimax=3e-3, slope=0.057), flag)
    u = pmx.GSTATE.FIELDX
    kw = dict(nspan=2, steps_per_span=4)
    gx, _ = _run(ctx, s, _cols(u), np.zeros_like(_cols(u)), bw, launches=1, gain_db=GAIN_DB, **kw)
    w = dbp_oracle.dbp_scalar(u, s.betat, s.gam, s.alphalin, s.nfc, s.length, s.fls[2], s.fls[3], gain=G16, bw=bw, **kw)
    err = np.linalg.norm(gx[0].T - w) / np.linalg.norm(w)
    print('filtered scalar dbp %s: %.3e' % (case, err))
    assert err <= 1e-10


@pytest.mark.gpu
@pytest.mark.parametrize('what', ['2pol_2e10', '2pol_2e14', 'scalar_ex06'])
def test_filtered_dbp_fp32(ctx, what):
    if what.startswith('scalar'):
        scalar_tx(32, 32, 1, pavg=1.0)       # the ex06 shape at the launch power of test_dbp_small's FP32 case (conditioning)
        s = fiber_setup(base_fiber(length=1e5, dphimax=3e-3, slope=0.057), 'g-sx')
        u = pmx.GSTATE.FIELDX
        gx, _ = _run(ctx, s, _cols(u), np.zeros_like(_cols(u)), 8.0, precision='f32', steps_per_span=4)
        w = dbp_oracle.dbp_scalar(u, s.betat, s.gam, s.alphalin, s.nfc, s.length, 1, 1, steps_per_span=4, bw=8.0)
        err = np.linalg.norm(gx[0].T - w) / np.linalg.norm(w)
    else:
        nsymb = 64 if what.endswith('2e10') else 1024
        gs, s = _setup(nsymb, 16, pavg_mw=4.0)
        gx, gy = _run(ctx, s, _cols(gs.FIELDX), _cols(gs.FIELDY), nsymb / 8.0, precision='f32', steps_per_span=4)
        err = rel_l2(gx[0].T, gy[0].T, *dbp_oracle.dbp(gs.FIELDX, gs.FIELDY, s.betat, s.gam, s.alphalin, 1, s.length, 'no',
                                                       steps_per_span=4, bw=nsymb / 8.0))
    print('filtered dbp fp32 %s: %.3e' % (what, err))
    assert err <= 1e-5


@pytest.mark.gpu
def test_filtered_dbp_c2_span(ctx):
    """one full C2 span (2^20 samples) on the three passes"""
    gs, s = _setup(65536, 16, pavg_mw=4.0, manakov=True)
    gx, gy = _run(ctx, s, _cols(gs.FIELDX), _cols(gs.FIELDY), 4096.0, steps_per_span=2)
    err = rel_l2(gx[0].T, gy[0].T, *dbp_oracle.dbp(gs.FIELDX, gs.FIELDY, s.betat, s.gam, s.alphalin, 1, s.length, 'yes',
                                                   steps_per_span=2, bw=4096.0))
    print('filtered dbp C2 span: %.3e' % err)
    assert err <= 1e-10


@pytest.mark.gpu
@pytest.mark.parametrize('nsymb,decim', [(1024, 16), (4096, 4)])
def test_single_channel_filtered_dbp_matches_the_oracle(ctx, nsymb, decim):
    """M = 2^10 (on-chip) and M = 2^14 (three passes)"""
    gs, s = _setup(nsymb, 16, pavg_mw=10.0)
    bw = s.nfft / decim / 8.0
    kw = dict(nspan=2, steps_per_span=2)
    gx, gy = _run(ctx, s, _cols(gs.FIELDX), _cols(gs.FIELDY), 0, gain_db=GAIN_DB, decim=decim, shift=0,
                  filter_bw=bw * pmx.GSTATE.SYMBOLRATE / pmx.GSTATE.NSYMB, **kw)
    wx, wy = dbp_oracle.dbp_channel(gs.FIELDX, gs.FIELDY, s.betat, s.gam, s.alphalin, s.length, 'no', 0, decim, gain=G16,
                                    bw=bw, **kw)
    err = rel_l2(gx[0].T, gy[0].T, wx, wy)
    print('filtered single-channel dbp 2^%d / %d: %.3e' % (int(np.log2(s.nfft)), decim, err))
    assert err <= 1e-10


@pytest.mark.gpu
@pytest.mark.parametrize('nsymb', [64, 1024])
def test_filter_plan_behaviour(ctx, nsymb):
    """set_filter(0) after a filtered run equals a fresh unfiltered plan bit for bit, a swapped bandwidth equals a fresh
    plan with it, and a batch of 5 equals each realization alone"""
    gs, s = _setup(nsymb, 16, pavg_mw=10.0)
    xs = np.concatenate([_cols(np.roll(gs.FIELDX, 13 * b, axis=0)) for b in range(5)])
    ys = np.concatenate([_cols(np.roll(gs.FIELDY, -3 * b, axis=0)) for b in range(5)])
    kw = dict(nspan=2, gain_db=GAIN_DB, steps_per_span=2, batch=5)
    fld = _lib.DeviceField(ctx, s.nfft, 1, 5)

    def run(plan):
        fld.upload(xs, ys)
        plan.execute(fld)
        return fld.download()
    plan = dbp_plan(ctx, s, **kw)
    plain = run(plan)
    plan.set_filter(nsymb / 4.0)
    f1 = run(plan)
    plan.set_filter(nsymb / 16.0)
    f2 = run(plan)
    plan.set_filter(0)
    back = run(plan)
    plan.close()
    fresh = dbp_plan(ctx, s, **kw)
    fresh.set_filter(nsymb / 16.0)
    f2_fresh = run(fresh)
    fresh.close()
    assert all(np.array_equal(a, b) for a, b in zip(back, plain))
    assert all(np.array_equal(a, b) for a, b in zip(f2, f2_fresh))
    assert not np.array_equal(f1[0], f2[0])
    fld.close()
    for b in range(5):
        ox, oy = _run(ctx, s, xs[b:b + 1], ys[b:b + 1], nsymb / 16.0, nspan=2, gain_db=GAIN_DB, steps_per_span=2)
        assert np.array_equal(ox[0], f2[0][b]) and np.array_equal(oy[0], f2[1][b]), b


@pytest.mark.gpu
def test_set_filter_rejects_on_real_plans(ctx):
    gs, s = _setup(64, 16)
    plan = dbp_plan(ctx, s)
    lib = _lib.load()
    assert lib.pmx_dbp_set_filter(plan.h, -2.0) == _lib.PMX_ERR_INVALID
    assert lib.pmx_dbp_set_filter(plan.h, float('nan')) == _lib.PMX_ERR_INVALID
    plan.close()
    from polmux_b200.fiber import setup_to_desc
    desc, keep = setup_to_desc(s)
    fp = _lib.Plan(ctx, desc, keep)
    assert lib.pmx_dbp_set_filter(fp.h, 2.0) == _lib.PMX_ERR_INVALID
    fp.close()


@pytest.mark.gpu
def test_pmx_dbp_filter_bw_end_to_end():
    gs, s = _setup(1024, 16, pavg_mw=10.0)
    G = pmx.GSTATE
    fib = base_fiber(length=8e4, slope=0.057, dphimax=0.02)
    x0, y0 = G.FIELDX.copy(), G.FIELDY.copy()
    pmx.dbp(fib, 'g-s-', nspan=2, gain_db=GAIN_DB, steps_per_span=2, filter_bw=5.0)
    bw = 5.0 * G.NSYMB / G.SYMBOLRATE
    wx, wy = dbp_oracle.dbp(x0, y0, s.betat, s.gam, s.alphalin, 1, s.length, 'no', nspan=2, gain=G16, steps_per_span=2,
                            bw=bw)
    err = rel_l2(G.FIELDX, G.FIELDY, wx, wy)
    print('pmx.dbp filter_bw: %.3e' % err)
    assert err <= 1e-10


# -------------------------------------------------------------------------------------------------- M front-end (dbp.m)
def test_m_front_end_sends_the_bandwidth_in_bins():
    """dbp.m with options.filter_bw: a 6-element D whose sixth entry is filter_bw*NSYMB/SYMBOLRATE, and the field of the
    filtered oracle on pmx.dbp's parameters"""
    import test_matlab_dbp as tmd
    make_tx(256, 16, pavg_mw=8.0)
    fib = base_fiber()
    G = pmx.GSTATE
    tx, ty = np.array(G.FIELDX), np.array(G.FIELDY)
    s = fiber_setup(fib, 'g-s-')
    bw = 7.0 * G.NSYMB / G.SYMBOLRATE
    want = dbp_oracle.dbp(tx, ty, s.betat, s.gam, s.alphalin, 1, s.length, 'no', nspan=2, gain=G16, steps_per_span=2,
                          bw=bw)
    gw = tmd.oracle_gateway()
    it = tmd._interp(gw)
    it.call('dbp', [tmd.to_m(fib), 'g-s-', tmd._opts(nspan=2, gain=GAIN_DB, steps=2, filter_bw=7.0)], 0)
    log = [e['D'] for e in gw.log if e['cmd'] == 'dbp']
    assert len(log) == 1 and log[0].size == 6 and log[0][5] == bw
    ux, uy = tmd._m_field(it)
    assert rel_l2(ux, uy, *want) <= 1e-13


@pytest.mark.gpu
def test_m_front_end_filtered_on_the_device():
    """dbp.m with filter_bw through the compiled gateway == pmx.dbp(..., filter_bw=) (on-chip and three passes)"""
    import test_matlab_dbp as tmd
    for nsymb in (64, 1024):
        make_tx(nsymb, 16, pavg_mw=8.0)
        m, p = tmd._device_pair(base_fiber(), 'g-s-', dict(nspan=2.0, gain=GAIN_DB, steps=2.0, filter_bw=6.0),
                                dict(nspan=2, gain_db=GAIN_DB, steps_per_span=2, filter_bw=6.0))
        assert tmd._err(m, p) <= 1e-13, nsymb


@pytest.mark.gpu
def test_mc_runner_with_filtered_dbp(ctx):
    """McRunner(compensation='dbp', dbp_params=dict(filter_bw=...)) runs with the 'cohmix' receiver; a very wide filter
    counts what plain DBP counts"""
    nsymb, nt, nspan, nreal, batch = 1 << 12, 16, 2, 8, 4
    G, setup, sym = _mc_scenario(nsymb, nt, 8.0)
    x = {'oftype': 'gauss', 'obw': 1.9, 'eftype': 'bessel5', 'ebw': 0.65, 'lopower': 0.0}
    counts = []
    for dp in (dict(steps_per_span=1), dict(steps_per_span=1, filter_bw=1e9), dict(steps_per_span=1, filter_bw=10.0)):
        r = mc.McRunner(ctx, setup, G.FIELDX_TX, G.FIELDY_TX, sym, nsymb, nt, nspan, 16.0, 5.0, nreal, batch,
                        receiver='cohmix', dsp_params=dict(mu=1 / 2000, freqavg=200), rx_params=x, compensation='dbp',
                        dbp_params=dp)
        c, _ = r.run(ase_seed=3)
        r.close()
        counts.append(c)
    print('McRunner filtered DBP counts: plain %s, wide %s, 10 GHz %s' % tuple(c.tolist() for c in counts))
    assert np.array_equal(counts[0], counts[1]) and counts[2].shape == (nreal,) and counts[2].min() >= 0
