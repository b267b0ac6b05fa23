"""Enhanced split-step digital backpropagation (pmx_dbp_set_taps, DbpPlan.set_taps, dbp_plan / pmx.dbp nl_taps, dbp.m
options.taps, tests/dbp_essfm_oracle.py): a circular FIR of real taps on the intensity of every backward nonlinear step."""
import numpy as np
import pytest

import dbp_essfm_oracle as deo
import dbp_filtered_oracle as dfo
import dbp_oracle
import dbp_scalar_oracle
import polmux_b200 as pmx
from polmux_b200 import _lib, mc
from polmux_b200.dbp import dbp_plan
from polmux_b200.fiber import fiber_setup
from common import base_fiber, make_tx, rel_l2, scalar_tx

GAIN_DB = 16.0
G16 = 10 ** (GAIN_DB / 10)


def taps(k, seed=0):
    """2k+1 real taps, sum 1, not symmetric (so that a lag of the wrong sign shows)"""
    m = np.arange(-k, k + 1, dtype=np.float64)
    c = np.exp(-(m / (0.5 * k + 1)) ** 2) * (1 + 0.2 * np.sin(m + seed))
    return c / c.sum() if k else np.array([0.8])


def _setup(nsymb, nt, nch=1, pavg_mw=4.0, manakov=False, flag='g-s-', length=8e4):
    gs = make_tx(nsymb, nt, nch=nch, ftype='sepfields' if nch > 1 else 'unique', pavg_mw=pavg_mw)
    s = fiber_setup(base_fiber(length=length, slope=0.057, dphimax=0.02), flag)
    s.manakov = manakov
    return gs, s


def _man(s):
    return 'yes' if s.manakov else 'no'


# ---------------------------------------------------------------------------------------------------------------- CPU
def _as_filtered(monkeypatch, nfft, c):
    """dbp_filtered_oracle with H = fft(c placed circularly) in place of its Gaussian (any bw selects it)"""
    monkeypatch.setattr(dfo, 'gauss_response', lambda n, bw: deo.circular_response(n, c))


@pytest.mark.parametrize('manakov', [False, True])
def test_oracle_is_filtered_dbp_with_the_circular_response_two_pol(monkeypatch, manakov):
    gs, s = _setup(64, 16, nch=3, pavg_mw=10.0, manakov=manakov)
    args = (gs.FIELDX, gs.FIELDY, s.betat, s.gam, s.alphalin, s.nfc, s.length, _man(s))
    kw = dict(nspan=2, gain=G16, steps_per_span=2)
    for k in (1, 16, 32):
        c = taps(k)
        a = deo.dbp(*args, taps=c, **kw)
        _as_filtered(monkeypatch, s.nfft, c)
        b = dfo.dbp(*args, bw=1.0, **kw)
        monkeypatch.undo()
        assert rel_l2(*a, *b) <= 1e-13, k
        assert rel_l2(*a, *deo.dbp(*args, **kw)) > 1e-6


def test_oracle_is_filtered_dbp_with_the_circular_response_pmd_and_channel(monkeypatch):
    gs = make_tx(64, 16, pavg_mw=10.0)
    s = fiber_setup(base_fiber(length=8e4, slope=0.057, dphimax=0.02, dgd=0.5, nplates=12, manakov='no'), 'gps-',
                    rng=np.random.Generator(np.random.PCG64(7)))
    brfs = [dict(zip(('db0', 'theta', 'epsilon'), mc.draw_plates(mc.plate_seed(0, k), s.nplates))) for k in range(2)]
    c = taps(7)
    kw = dict(nspan=2, gain=G16, steps_per_span=2)
    pargs = (gs.FIELDX, gs.FIELDY, s.betat, np.asarray(s.db1), s.gam, s.alphalin, 1, s.length, 'no', brfs)
    a = deo.dbp_pmd(*pargs, taps=c, **kw)
    cargs = (gs.FIELDX, gs.FIELDY, s.betat, s.gam, s.alphalin, s.length, 'no', 0, 4)
    ca = deo.dbp_channel(*cargs, taps=c, **kw)
    _as_filtered(monkeypatch, s.nfft, c)
    assert rel_l2(*a, *dfo.dbp_pmd(*pargs, bw=1.0, **kw)) <= 1e-13
    monkeypatch.setattr(dfo, 'gauss_response', lambda n, bw: deo.circular_response(n, c))   # (on the channel's grid)
    assert rel_l2(*ca, *dfo.dbp_channel(*cargs, bw=1.0, **kw)) <= 1e-13


@pytest.mark.parametrize('flag', ['g-s-', 'g--x', 'g-sx'])
def test_oracle_is_filtered_dbp_with_the_circular_response_scalar(monkeypatch, flag):
    u = scalar_tx(32, 32, 3, pavg=8.0).FIELDX
    ss = fiber_setup(base_fiber(length=1e5, slope=0.057), flag)
    sa = (u, ss.betat, ss.gam, ss.alphalin, ss.nfc, ss.length, ss.fls[2], ss.fls[3])
    kw = dict(nspan=2, gain=G16, steps_per_span=3)
    c = taps(5)
    a = deo.dbp_scalar(*sa, taps=c, **kw)
    _as_filtered(monkeypatch, u.shape[0], c)
    b = dfo.dbp_scalar(*sa, bw=1.0, **kw)
    assert np.linalg.norm(a - b) <= 1e-13 * np.linalg.norm(b)


def test_oracle_single_unit_tap_is_plain_dbp():
    gs, s = _setup(64, 16, nch=2, pavg_mw=10.0)
    args = (gs.FIELDX, gs.FIELDY, s.betat, s.gam, s.alphalin, s.nfc, s.length, 'no')
    kw = dict(nspan=2, gain=G16, steps_per_span=3)
    assert rel_l2(*deo.dbp(*args, taps=[1.0], **kw), *dbp_oracle.dbp(*args, **kw)) <= 1e-14
    u = scalar_tx(32, 32, 3, pavg=8.0).FIELDX
    ss = fiber_setup(base_fiber(length=1e5, slope=0.057), 'g-sx')
    sa = (u, ss.betat, ss.gam, ss.alphalin, ss.nfc, ss.length, 1, 1)
    a = deo.dbp_scalar(*sa, taps=[1.0], **kw)
    b = dbp_scalar_oracle.dbp_scalar(*sa, **kw)
    assert np.linalg.norm(a - b) <= 1e-14 * np.linalg.norm(b)


def test_set_taps_rejects_without_a_context():
    lib = _lib.load()
    for c in ([0.5, 0.5], list(np.ones(67) / 67), [0.2, float('nan'), 0.2], [0.2, float('inf'), 0.2]):
        a = np.asarray(c, dtype=np.float64)
        assert lib.pmx_dbp_set_taps(None, a.size, a.ctypes.data_as(_lib._dp)) == _lib.PMX_ERR_INVALID
        with pytest.raises(ValueError, match='pmx_dbp_set_taps'):
            _lib.check_taps(a)
    assert lib.pmx_dbp_set_taps(None, -1, None) == _lib.PMX_ERR_INVALID
    assert lib.pmx_dbp_set_taps(None, 3, None) == _lib.PMX_ERR_INVALID
    make_tx(64, 16)
    fib = base_fiber()
    with pytest.raises(ValueError, match='ntaps must be odd and at most 65 .0: no taps., got 2'):
        pmx.dbp(fib, 'g-s-', nl_taps=[0.5, 0.5])
    with pytest.raises(ValueError, match='tap 1 is not finite'):
        pmx.dbp(fib, 'g-s-', nl_taps=[0.2, float('nan'), 0.2])
    with pytest.raises(ValueError, match='a plan takes one or the other'):
        pmx.dbp(fib, 'g-s-', nl_taps=[1.0], filter_bw=5.0)


def test_native_mc_rejects_nl_taps():
    s = fiber_setup(base_fiber(), 'g-s-')
    with pytest.raises(ValueError, match='nl_taps'):
        mc.run_mc_native(s, None, None, None, 16, 16, 1, 16.0, 5.0, 1, 1, receiver={}, dbp_params=dict(nl_taps=[1.0]))


# -------------------------------------------------------------------------------------------------- M front-end (dbp.m)
def _taps_gateway(log):
    """test_matlab_dbp's oracle-backed gateway; a 'dbp' call with the trailing taps (two polarizations, full field, no PMD)
    is answered by the ESSFM oracle.  Every 'dbp' call logs its taps (None: the 15-argument call)."""
    import test_matlab_dbp as tmd
    base = tmd.oracle_gateway()

    def call(it, a, nargout):
        if a[0] != 'dbp':
            return base(it, a, nargout)
        log.append(np.asarray(a[15], dtype=np.float64) if len(a) > 15 else None)
        if len(a) == 15:
            return base(it, a, nargout)
        assert len(a) == 16 and np.size(a[15]) > 0
        ux, uy, betat, db1, P, gam = a[1:7]
        scal, D, fls = a[9], np.asarray(a[10], dtype=np.float64).ravel(), [int(v) for v in np.asarray(a[7]).ravel()]
        _, _, alphalin, lf, _, manakov = [float(v) for v in np.asarray(P).ravel()]
        nfft, nfc = np.shape(ux)
        if np.size(betat) == 0:
            betat, db1 = tmd._vectors(scal, nfft, nfc, fls[1])
        out = deo.dbp(ux, uy, betat, np.asarray(gam, dtype=np.float64).ravel(), alphalin, nfc, lf,
                      'yes' if manakov else 'no', spm=fls[2], nspan=int(D[0]), gain=D[1] or None,
                      steps_per_span=int(D[2]), xi=D[3], taps=np.asarray(a[15], dtype=np.float64).ravel())
        return list(out)[:max(nargout, 1)]
    return call


@pytest.mark.parametrize('shape', ['row', 'column'])
def test_m_front_end_sends_the_taps(shape):
    """dbp.m with options.taps (a row or a column): the gateway's trailing argument, and the field of the ESSFM oracle on
    pmx.dbp's parameters; without taps the call keeps its 15 arguments"""
    import test_matlab_dbp as tmd
    make_tx(256, 16, pavg_mw=8.0)
    fib = base_fiber()
    G = pmx.GSTATE
    tx, ty = np.array(G.FIELDX), np.array(G.FIELDY)
    s = fiber_setup(fib, 'g-s-')
    c = taps(3)
    want = deo.dbp(tx, ty, s.betat, s.gam, s.alphalin, 1, s.length, 'no', nspan=2, gain=G16, steps_per_span=2, taps=c)
    log = []
    it = tmd._interp(_taps_gateway(log))
    m = c.reshape(1, -1) if shape == 'row' else c.reshape(-1, 1)
    it.call('dbp', [tmd.to_m(fib), 'g-s-', tmd._opts(nspan=2, gain=GAIN_DB, steps=2, taps=m)], 0)
    assert len(log) == 1 and np.array_equal(log[0].ravel(), c)
    assert rel_l2(*tmd._m_field(it), *want) <= 1e-13
    it.call('dbp', [tmd.to_m(fib), 'g-s-', tmd._opts(nspan=2, gain=GAIN_DB, steps=2, taps=np.zeros((0, 0)))], 0)
    assert len(log) == 2 and log[1] is None


@pytest.mark.parametrize('case', ['even', 'too_many', 'nan', 'with_filter_bw'])
def test_m_front_end_refusals_are_pmx_dbp_s(case):
    import test_matlab_dbp as tmd
    make_tx(256, 16)
    fib = base_fiber()
    c, extra = {'even': (np.ones(4) / 4, {}), 'too_many': (np.ones(67) / 67, {}),
                'nan': (np.array([0.1, 0.8, np.nan]), {}), 'with_filter_bw': (np.array([1.0]), dict(filter_bw=5.0))}[case]
    want = tmd._python_error(lambda: pmx.dbp(fib, 'g-s-', nl_taps=c, **extra))
    it = tmd._interp(tmd.oracle_gateway())
    with pytest.raises(tmd.MError) as e:
        it.call('dbp', [tmd.to_m(fib), 'g-s-', tmd._opts(taps=c.reshape(1, -1), **extra)], 0)
    assert str(e.value) == want


# ---------------------------------------------------------------------------------------------------------------- GPU
def _cols(a):
    return np.ascontiguousarray(np.asarray(a).T)[None]


def _run(ctx, s, xs, ys, c, precision='f64', plates=None, **kw):
    b = xs.shape[0]
    fld = _lib.DeviceField(ctx, s.nfft, s.nfc, b, precision={'f64': _lib.PMX_F64, 'f32': _lib.PMX_F32}[precision])
    fld.upload(xs, ys)
    plan = dbp_plan(ctx, s, batch=b, precision=precision, plates=plates, nl_taps=c, **kw)
    plan.execute(fld)
    plan.close()
    out = fld.download()
    fld.close()
    return out


def _two_pol(ctx, nsymb, nt, nch, manakov, batch, k, steps=2, nspan=2, precision='f64'):
    gs, s = _setup(nsymb, nt, nch=nch, pavg_mw=10.0, manakov=manakov)
    xs = np.concatenate([_cols(np.roll(gs.FIELDX, 7 * b, axis=0)) for b in range(batch)])
    ys = np.concatenate([_cols(np.roll(gs.FIELDY, -5 * b, axis=0)) for b in range(batch)])
    kw = dict(nspan=nspan, steps_per_span=steps)
    c = taps(k)
    gx, gy = _run(ctx, s, xs, ys, c, precision=precision, gain_db=GAIN_DB, **kw)
    errs = []
    for b in range(batch):
        wx, wy = deo.dbp(xs[b].T, ys[b].T, s.betat, s.gam, s.alphalin, s.nfc, s.length, _man(s), gain=G16, taps=c, **kw)
        errs.append(rel_l2(gx[b].T, gy[b].T, wx, wy))
    return errs


@pytest.mark.gpu
@pytest.mark.parametrize('k', [0, 1, 16, 32])
@pytest.mark.parametrize('nsymb,batch', [(256, 3), (4096, 2), (65536, 2)], ids=['2e12', '2e16', '2e20'])
def test_three_pass_essfm_matches_the_oracle(ctx, nsymb, batch, k):
    """2^12 (N1 = N2 = 64: k = 32 reaches across the row wrap), 2^16 and 2^20; Manakov at even k, CNLSE at odd"""
    steps, nspan = (1, 1) if nsymb == 65536 else (2, 2)
    errs = _two_pol(ctx, nsymb, 16, 1, k % 2 == 0, batch, k, steps=steps, nspan=nspan)
    print('essfm three passes %d x 16, k %d: %s' % (nsymb, k, ['%.3e' % e for e in errs]))
    assert max(errs) <= 1e-10


@pytest.mark.gpu
@pytest.mark.parametrize('k', [0, 1, 16, 32])
@pytest.mark.parametrize('nsymb,nch,batch', [(4, 1, 2), (64, 1, 3), (128, 3, 1)], ids=['2e6', '2e10', '2e11x3'])
def test_on_chip_essfm_matches_the_oracle(ctx, nsymb, nch, batch, k):
    k = min(k, 31) if nsymb == 4 else k   # 2^6 samples take at most 63 taps
    errs = _two_pol(ctx, nsymb, 16, nch, k % 2 == 1, batch, k)
    print('essfm on-chip %d x 16 x %d, k %d: %s' % (nsymb, nch, k, ['%.3e' % e for e in errs]))
    assert max(errs) <= 1e-10


SCALAR = [  # nsymb, nt, nch, flag, k
    (32, 32, 8, 'g-sx', 16),     # 2^10, eight columns
    (32, 32, 8, 'g-sx', 32),
    (128, 32, 3, 'g-sx', 32),    # 2^12: the resident column is transposed
    (128, 32, 1, 'g-s-', 1),
]


@pytest.mark.gpu
@pytest.mark.parametrize('case', SCALAR, ids=lambda c: '%dx%dx%d-%s-k%d' % c)
def test_scalar_essfm_matches_the_oracle(ctx, case):
    nsymb, nt, nch, flag, k = case
    scalar_tx(nsymb, nt, nch, pavg=8.0)
    s = fiber_setup(base_fiber(length=1e5, dphimax=3e-3, slope=0.057), flag)
    u = pmx.GSTATE.FIELDX
    kw = dict(nspan=2, steps_per_span=3)
    c = taps(k, seed=2)
    gx, _ = _run(ctx, s, _cols(u), np.zeros_like(_cols(u)), c, gain_db=GAIN_DB, **kw)
    w = deo.dbp_scalar(u, s.betat, s.gam, s.alphalin, s.nfc, s.length, s.fls[2], s.fls[3], gain=G16, taps=c, **kw)
    err = np.linalg.norm(gx[0].T - w) / np.linalg.norm(w)
    print('essfm scalar %s: %.3e' % (case, err))
    assert err <= 1e-10


@pytest.mark.gpu
@pytest.mark.parametrize('nsymb', [64, 1024])
def test_pmd_essfm_matches_the_oracle(ctx, nsymb):
    """PMD-aware, per-realization plates: on-chip (2^10) and three passes (2^14)"""
    gs = make_tx(nsymb, 16, pavg_mw=10.0)
    s = fiber_setup(base_fiber(length=8e4, slope=0.057, dphimax=0.02, dgd=0.5, nplates=12, manakov='no'), 'gps-',
                    rng=np.random.Generator(np.random.PCG64(7)))
    nspan, batch, c = 2, 2, taps(16)
    brfs = [[dict(zip(('db0', 'theta', 'epsilon'), mc.draw_plates(mc.plate_seed(b, k), s.nplates))) for k in range(nspan)]
            for b in range(batch)]
    plates = tuple(np.array([[brfs[b][k][n] for b in range(batch)] for k in range(nspan)])
                   for n in ('db0', 'theta', 'epsilon'))
    xs = np.concatenate([_cols(np.roll(gs.FIELDX, 9 * b, axis=0)) for b in range(batch)])
    ys = np.concatenate([_cols(gs.FIELDY) for b in range(batch)])
    kw = dict(nspan=nspan, steps_per_span=2)
    gx, gy = _run(ctx, s, xs, ys, c, plates=plates, gain_db=GAIN_DB, **kw)
    for b in range(batch):
        wx, wy = deo.dbp_pmd(xs[b].T, ys[b].T, s.betat, np.asarray(s.db1), s.gam, s.alphalin, 1, s.length, 'no', brfs[b],
                             gain=G16, taps=c, **kw)
        err = rel_l2(gx[b].T, gy[b].T, wx, wy)
        print('essfm pmd 2^%d b%d: %.3e' % (int(np.log2(s.nfft)), b, err))
        assert err <= 1e-10


@pytest.mark.gpu
def test_single_channel_essfm_matches_the_oracle(ctx):
    """N = 2^16, r = 16: the taps act on the channel's 2^12 samples (three passes)"""
    gs, s = _setup(4096, 16, pavg_mw=10.0)
    c, kw = taps(16), dict(nspan=2, steps_per_span=2)
    gx, gy = _run(ctx, s, _cols(gs.FIELDX), _cols(gs.FIELDY), c, gain_db=GAIN_DB, decim=16, shift=0, **kw)
    wx, wy = deo.dbp_channel(gs.FIELDX, gs.FIELDY, s.betat, s.gam, s.alphalin, s.length, 'no', 0, 16, gain=G16, taps=c,
                             **kw)
    err = rel_l2(gx[0].T, gy[0].T, wx, wy)
    print('essfm single-channel 2^16 / 16: %.3e' % err)
    assert err <= 1e-10


@pytest.mark.gpu
@pytest.mark.parametrize('nsymb', [64, 1024])
def test_essfm_fp32(ctx, nsymb):
    errs = _two_pol(ctx, nsymb, 16, 1, False, 2, 16, precision='f32')
    print('essfm fp32 %d x 16: %s' % (nsymb, ['%.3e' % e for e in errs]))
    assert max(errs) <= 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize('nsymb', [64, 4096])
def test_essfm_plan_behaviour(ctx, nsymb):
    """two runs are bitwise equal; set_taps([]) after an ESSFM run equals a fresh plain plan bit for bit; swapped taps equal
    a fresh plan with them"""
    gs, s = _setup(nsymb, 16, pavg_mw=10.0)
    xs = np.concatenate([_cols(np.roll(gs.FIELDX, 13 * b, axis=0)) for b in range(3)])
    ys = np.concatenate([_cols(np.roll(gs.FIELDY, -3 * b, axis=0)) for b in range(3)])
    kw = dict(nspan=2, gain_db=GAIN_DB, steps_per_span=2, batch=3)
    fld = _lib.DeviceField(ctx, s.nfft, 1, 3)

    def run(plan):
        fld.upload(xs, ys)
        plan.execute(fld)
        return fld.download()
    plan = dbp_plan(ctx, s, **kw)
    plain = run(plan)
    plan.set_taps(taps(16))
    e1 = run(plan)
    e1b = run(plan)
    plan.set_taps(taps(3))
    e2 = run(plan)
    plan.set_taps([])
    back = run(plan)
    plan.close()
    fresh = dbp_plan(ctx, s, nl_taps=taps(3), **kw)
    e2_fresh = run(fresh)
    fresh.close()
    fld.close()
    assert all(np.array_equal(a, b) for a, b in zip(e1, e1b))
    assert all(np.array_equal(a, b) for a, b in zip(back, plain))
    assert all(np.array_equal(a, b) for a, b in zip(e2, e2_fresh))
    assert not np.array_equal(e1[0], e2[0]) and not np.array_equal(e1[0], plain[0])


@pytest.mark.gpu
def test_set_taps_rejects_on_real_plans(ctx):
    lib = _lib.load()
    gs, s = _setup(4, 16)   # 2^6 samples
    one = np.array([1.0])
    t65 = np.ones(65) / 65
    plan = dbp_plan(ctx, s)
    assert lib.pmx_dbp_set_taps(plan.h, 65, t65.ctypes.data_as(_lib._dp)) == _lib.PMX_ERR_INVALID   # more taps than samples
    assert lib.pmx_dbp_set_taps(plan.h, 63, t65.ctypes.data_as(_lib._dp)) == _lib.PMX_OK
    assert lib.pmx_dbp_set_filter(plan.h, 4.0) == _lib.PMX_ERR_INVALID    # taps, then a bandwidth
    assert lib.pmx_dbp_set_filter(plan.h, 0.0) == _lib.PMX_OK
    assert lib.pmx_dbp_set_taps(plan.h, 0, None) == _lib.PMX_OK
    assert lib.pmx_dbp_set_filter(plan.h, 4.0) == _lib.PMX_OK
    assert lib.pmx_dbp_set_taps(plan.h, 1, one.ctypes.data_as(_lib._dp)) == _lib.PMX_ERR_INVALID   # a bandwidth, then taps
    plan.close()
    from polmux_b200.fiber import setup_to_desc
    desc, keep = setup_to_desc(s)
    fp = _lib.Plan(ctx, desc, keep)
    assert lib.pmx_dbp_set_taps(fp.h, 1, one.ctypes.data_as(_lib._dp)) == _lib.PMX_ERR_INVALID
    fp.close()


@pytest.mark.gpu
def test_m_front_end_essfm_on_the_device():
    """dbp.m with options.taps through the compiled gateway == pmx.dbp(..., nl_taps=) (on-chip and three passes)"""
    import test_matlab_dbp as tmd
    c = taps(16)
    for nsymb in (64, 1024):
        make_tx(nsymb, 16, pavg_mw=8.0)
        m, p = tmd._device_pair(base_fiber(), 'g-s-', dict(nspan=2.0, gain=GAIN_DB, steps=2.0, taps=c.reshape(1, -1)),
                                dict(nspan=2, gain_db=GAIN_DB, steps_per_span=2, nl_taps=c))
        assert tmd._err(m, p) == 0.0, nsymb


@pytest.mark.gpu
def test_mc_runner_with_essfm(ctx):
    """McRunner(compensation='dbp', dbp_params=dict(nl_taps=[1.0])) counts what plain DBP counts, behind the 'cohmix' and
    the 'blind' receiver"""
    import test_dbp as td
    nsymb, nt, nspan, nreal, batch = 1 << 12, 16, 2, 8, 4
    G, setup, sym = td._mc_scenario(nsymb, nt, 8.0)
    x = {'oftype': 'gauss', 'obw': 1.9, 'eftype': 'bessel5', 'ebw': 0.65, 'lopower': 0.0}
    for receiver in ('cohmix', 'blind'):
        counts = []
        for dp in (dict(steps_per_span=1), dict(steps_per_span=1, nl_taps=[1.0])):
            kw = dict(rx_params=x) if receiver == 'cohmix' else {}
            r = mc.McRunner(ctx, setup, G.FIELDX_TX, G.FIELDY_TX, sym, nsymb, nt, nspan, 16.0, 5.0, nreal, batch,
                            receiver=receiver, dsp_params=dict(mu=1 / 2000, freqavg=200), compensation='dbp',
                            dbp_params=dp, **kw)
            c, _ = r.run(ase_seed=3)
            r.close()
            counts.append(c)
        print('McRunner essfm %s counts: plain %s, one unit tap %s' % (receiver, *[c.tolist() for c in counts]))
        assert np.array_equal(counts[0], counts[1])
