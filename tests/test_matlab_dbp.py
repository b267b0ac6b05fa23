"""matlab/dbp.m -- the M front-end of digital backpropagation -- and the gateway command ssfm_mex('dbp', ...), executed
by the mini M interpreter (oracle/mini_m).

CPU: dbp.m with a gateway whose 'dbp' command is served by the DBP oracles (tests/dbp_oracle.py, dbp_pmd_oracle.py,
dbp_scalar_oracle.py, dbp_channel_oracle.py) equals those oracles run on the parameters the Python mirror pmx.dbp derives
from the same GSTATE; a PMD-aware DBP inverts two 'gps-' spans that the interpreted fiber.m + ampliflat.m ran; every
refusal of dbp.m carries pmx.dbp's message.
GPU: the same front-end with the compiled gateway (mexFunction of mex/ssfm_mex.c through the mex.h stand-in) equals
pmx.dbp on every route, keeps the field resident after fiber.m / ampliflat.m, and inverts a link that fiber.m ran."""
import math
import os

import numpy as np
import pytest

import oracle.fiber_oracle as orc
from oracle.mini_m.interp import Interp, MCell, MError, MStruct, to_m
import dbp_channel_oracle as dco
import dbp_oracle
import dbp_pmd_oracle
import dbp_scalar_oracle
import mex_bridge
import polmux_b200 as pmx
from common import base_fiber, make_tx, rel_l2, scalar_tx

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MDIR = os.path.join(ROOT, 'matlab')
GAIN_DB = 16.0


# ------------------------------------------------------------------------------------------------------------ fixtures
def _vectors(scal, nfft, nfc, pflag):
    """betat / db1 of the scalar dispersion mode (fiber.m:350-362 from the scalars), as the library rebuilds them"""
    s = np.asarray(scal, dtype=np.float64).ravel()
    rate, nsymb, nt, b30, dgdrms = s[:5]
    b1, b2 = s[5:5 + nfc], s[5 + nfc:5 + 2 * nfc]
    omega = 2 * math.pi * rate * np.fft.fftshift(-nt / 2.0 + np.arange(nfft) / nsymb)
    betat = np.stack([omega * b1[k] + 0.5 * omega ** 2 * b2[k] + omega ** 3 * b30 / 6 for k in range(nfc)], axis=1)
    return betat, np.stack([dgdrms * omega * (1 if pflag else 0) for _ in range(nfc)], axis=1)


def oracle_gateway(log=None):
    """mex_bridge.oracle_gateway() plus ssfm_mex('dbp', ...) answered by the DBP oracles.  Every 'dbp' call is logged
    (its P, fls, D, band, opt); every two-polarization 'fiber' call logs the oracle's forward steps."""
    base = mex_bridge.oracle_gateway()
    log = [] if log is None else log

    def call(it, a, nargout):
        if a[0] == 'fiber' and not (len(a) > 10 and np.size(a[10]) and float(np.asarray(a[10]).ravel()[0])):
            ux, uy, betat, db1, P, gam, fls, plates, scal = a[1:10]
            dzmaxt, dphimaxt, alphalin, lf, nplates, manakov = [float(v) for v in np.asarray(P).ravel()]
            fls = [int(v) for v in np.asarray(fls).ravel()]
            nfft, nfc = np.shape(ux)
            if np.size(betat) == 0:
                betat, db1 = _vectors(scal, nfft, nfc, fls[1])
            pl = np.asarray(plates, dtype=np.float64)
            brf = ({'db0': pl[:, 0], 'theta': pl[:, 1], 'epsilon': pl[:, 2]} if pl.size
                   else {'db0': np.zeros(1), 'theta': np.zeros(1), 'epsilon': np.zeros(1)})
            firstdz, ncycle, x1, y1, _, sched = orc.matrix_ssfm(ux, uy, betat, db1, dzmaxt, dphimaxt, np.asarray(gam).ravel(),
                                                                alphalin, nfc, lf, int(nplates), 'yes' if manakov else 'no',
                                                                fls, brf)
            log.append(dict(cmd='fiber', steps=[st['dz'] for st in sched]))
            return [x1, y1, np.array([[float(firstdz)]]), np.array([[float(ncycle)]])][:max(nargout, 1)]
        if a[0] != 'dbp':
            return base(it, a, nargout)
        ux, uy, betat, db1, P, gam, fls, plates, scal, D, steplen, spansteps, band, opt = a[1:15]
        dzmaxt, dphimaxt, alphalin, lf, nplates, manakov = [float(v) for v in np.asarray(P).ravel()]
        fls = [int(v) for v in np.asarray(fls).ravel()]
        nspan, gain, steps, xi, pmd = [float(v) for v in np.asarray(D).ravel()]
        opt = np.asarray(opt, dtype=np.float64).ravel()
        log.append(dict(cmd='dbp', P=np.asarray(P).ravel(), fls=fls, D=np.asarray(D).ravel(), band=np.asarray(band).ravel(),
                        opt=opt, scal=np.asarray(scal).ravel(), gam=np.asarray(gam).ravel()))
        nfft, nfc = np.shape(ux)
        if np.size(betat) == 0:
            betat, db1 = _vectors(scal, nfft, nfc, fls[1])
        nspan = int(nspan)
        kw = dict(nspan=nspan, gain=gain if gain else None, xi=xi)
        if steps:
            kw['steps_per_span'] = int(steps)
        else:
            kw['step_len'] = np.asarray(steplen, dtype=np.float64).ravel()
            kw['span_steps'] = [int(v) for v in np.asarray(spansteps).ravel()] if np.size(spansteps) else None
        gam = np.asarray(gam, dtype=np.float64).ravel()
        mk = 'yes' if manakov else 'no'
        ch = np.size(band) != 0
        shift, decim = ([int(v) for v in np.asarray(band).ravel()] if ch else (0, 1))
        if opt[0]:                                         # the scalar path
            if ch:
                out = dco.dbp_channel_scalar(ux, betat, gam, alphalin, lf, shift, decim, spm=fls[2], **kw)
            else:
                out = dbp_scalar_oracle.dbp_scalar(ux, betat, gam, alphalin, nfc, lf, spm=fls[2], xpm=fls[3], **kw)
            return [out, np.zeros((0, 0))][:max(nargout, 1)]
        brfs = None
        if pmd:
            pl = np.asarray(plates, dtype=np.float64)
            n = int(nplates)
            brfs = [{'db0': pl[k * n:(k + 1) * n, 0], 'theta': pl[k * n:(k + 1) * n, 1],
                     'epsilon': pl[k * n:(k + 1) * n, 2]} for k in range(nspan)]
        if ch:
            ox, oy = dco.dbp_channel(ux, uy, betat, gam, alphalin, lf, mk, shift, decim, db1=db1, brfs=brfs, spm=fls[2], **kw)
        elif pmd:
            ox, oy = dbp_pmd_oracle.dbp_pmd(ux, uy, betat, db1, gam, alphalin, nfc, lf, mk, brfs, spm=fls[2], **kw)
        else:
            ox, oy = dbp_oracle.dbp(ux, uy, betat, gam, alphalin, nfc, lf, mk, spm=fls[2], **kw)
        return [ox, oy][:max(nargout, 1)]
    call.log = log
    return call


def _m_globals(it, pmxopt=None):
    """the interpreter's GSTATE / CONSTANTS <- the product's GSTATE (what reset_all.m + create_field.m leave)"""
    G = pmx.GSTATE
    it.globals['CONSTANTS'] = MStruct({'CLIGHT': to_m(orc.CLIGHT), 'HPLANCK': to_m(orc.HPLANCK),
                                       'ECHARGE': to_m(orc.ECHARGE), 'KBOLTZMANN': to_m(orc.KBOLTZMANN)})
    nch = int(G.NCH)
    two = G.has_y()
    it.globals['GSTATE'] = MStruct({
        'NSYMB': to_m(G.NSYMB), 'NT': to_m(G.NT), 'NCH': to_m(nch), 'FN': np.asarray(G.FN, dtype=np.float64).reshape(1, -1),
        'SYMBOLRATE': to_m(float(G.SYMBOLRATE)), 'LAMBDA': np.asarray(G.LAMBDA, dtype=np.float64).reshape(1, -1),
        'POWER': np.asarray(G.POWER, dtype=np.float64).reshape(1, -1), 'FIELDX': np.array(G.FIELDX),
        'FIELDY': np.array(G.FIELDY) if two else np.zeros((0, 0)),
        'DELAY': np.zeros((2 if two else 1, nch)), 'DISP': np.zeros((2 if two else 1, nch)),
        'PRINT': np.array([[False]]), 'DIR': 'sim'})
    it.globals['PMXOPT'] = MStruct({k: (v if isinstance(v, str) else to_m(v)) for k, v in (pmxopt or {}).items()})


def _interp(gw, seed=0, pmxopt=None):
    it = Interp([MDIR], rng=np.random.Generator(np.random.PCG64(seed)))
    it.builtins['ssfm_mex'] = gw
    _m_globals(it, pmxopt)
    return it


def _opts(**kw):
    return MStruct({k: (v if isinstance(v, (str, MCell, MStruct)) else to_m(v)) for k, v in kw.items()})


def _brf_m(b):
    return MStruct({k: np.asarray(b[k], dtype=np.float64).reshape(-1, 1) for k in ('db0', 'theta', 'epsilon')})


def _rel(a, b):
    return float(np.linalg.norm(np.asarray(a) - np.asarray(b)) / np.linalg.norm(np.asarray(b)))


def _m_field(it):
    G = it.globals['GSTATE']
    return np.asarray(G['FIELDX']), np.asarray(G['FIELDY'])


def _setup(fib, flag):
    """pmx.dbp's FiberSetup of the same fiber on the product's GSTATE (the 'p' flag dropped, as without brf)"""
    f = flag.lower()
    return pmx.fiber_setup(fib, f[0] + '-' + f[2:])


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_two_polarizations_manakov_uniform_steps_with_gain():
    """'gps-' with x.manakov = 'yes' and no brf: the 'p' flag is dropped (no draw), the model stays Manakov; 2 spans,
    16 dB, 3 steps per span == dbp_oracle on pmx.dbp's parameters"""
    make_tx(256, 16, pavg_mw=4.0)
    fib = base_fiber(dgd=0.5, nplates=20, manakov='yes')
    G = pmx.GSTATE
    tx, ty = np.array(G.FIELDX), np.array(G.FIELDY)
    s = _setup(fib, 'gps-')
    want = dbp_oracle.dbp(tx, ty, s.betat, s.gam, s.alphalin, 1, s.length, 'yes', nspan=2, gain=10 ** (GAIN_DB / 10),
                          steps_per_span=3)
    gw = oracle_gateway()
    it = _interp(gw, seed=3)
    state = it.rng.bit_generator.state
    it.call('dbp', [to_m(fib), 'gps-', _opts(nspan=2, gain=GAIN_DB, steps=3)], 0)
    assert it.rng.bit_generator.state == state                  # nothing taken from the rand stream
    ux, uy = _m_field(it)
    assert rel_l2(ux, uy, *want) <= 1e-13
    c = gw.log[-1]
    assert c['fls'] == [1, 0, 1, 0] and c['P'][5] == 1 and c['P'][4] == 1 and list(c['opt']) == [0, 0, 1]
    assert list(c['D']) == [2, 10 ** (GAIN_DB / 10), 3, 1, 0] and c['band'].size == 0
    G = it.globals['GSTATE']
    assert not np.any(G['DELAY']) and not np.any(G['DISP'])    # DELAY / DISP untouched


def test_explicit_schedule():
    """steplen + spansteps (every span its own steps) and steplen alone (one span's steps, every span) == the oracle"""
    make_tx(256, 16, pavg_mw=4.0)
    fib = base_fiber()
    G = pmx.GSTATE
    tx, ty = np.array(G.FIELDX), np.array(G.FIELDY)
    s = _setup(fib, 'g-s-')
    L = s.length
    steps = np.array([0.1, 0.2, 0.7, 0.25, 0.25, 0.25, 0.25]) * L
    for sl, ss in ((steps, [3, 4]), (steps[:3], None)):
        want = dbp_oracle.dbp(tx, ty, s.betat, s.gam, s.alphalin, 1, L, 'no', nspan=2, gain=10 ** (GAIN_DB / 10),
                              step_len=sl, span_steps=ss, xi=0.7)
        it = _interp(oracle_gateway())
        o = dict(nspan=2, gain=GAIN_DB, steplen=sl.reshape(1, -1), xi=0.7)
        if ss:
            o['spansteps'] = np.array([ss], dtype=np.float64)
        it.call('dbp', [to_m(fib), 'g-s-', _opts(**o)], 0)
        assert rel_l2(*_m_field(it), *want) <= 1e-13
    with pytest.raises(MError, match='give steps_per_span or step_len, not both'):        # (as polmux_b200._lib.make_dbp)
        it.call('dbp', [to_m(fib), 'g-s-', _opts(steps=2.0, steplen=np.array([[L]]))], 0)


def test_scalar_xpm_sepfields_ex10_shape():
    """scalar 'g-sx' on 5 'sepfields' columns of 2^11 samples: XPM-aware DBP == dbp_scalar_oracle; FIELDY stays empty"""
    scalar_tx(64, 32, 5)
    fib = base_fiber(length=5e4)
    G = pmx.GSTATE
    tx = np.array(G.FIELDX)
    s = _setup(fib, 'g-sx')
    assert s.fls[3] == 1 and not s.isv
    want = dbp_scalar_oracle.dbp_scalar(tx, s.betat, s.gam, s.alphalin, 5, s.length, spm=1, xpm=1, nspan=2,
                                        gain=10 ** (GAIN_DB / 10), steps_per_span=4)
    gw = oracle_gateway()
    it = _interp(gw)
    it.call('dbp', [to_m(fib), 'g-sx', _opts(nspan=2, gain=GAIN_DB, steps=4)], 0)
    ux, uy = _m_field(it)
    assert uy.size == 0 and ux.shape == tx.shape
    assert _rel(ux, want) <= 1e-13
    assert gw.log[-1]['opt'][0] == 1 and gw.log[-1]['fls'] == [1, 0, 1, 1]
    np.testing.assert_array_equal(gw.log[-1]['gam'], s.gam)                   # fiber.m's gamma per column


def test_pmd_aware_inverts_two_spans_of_the_interpreted_fiber():
    """two noise-free 'gps-' spans through the interpreted matlab/fiber.m + ampliflat.m (other plates in every span,
    brf returned by fiber.m), then dbp.m with the cell of both brf, xi = 1 and the oracle's forward steps: the Tx field
    back to <= 1e-12, and == dbp_pmd_oracle"""
    make_tx(256, 16, pavg_mw=4.0)
    fib = base_fiber(dgd=0.5, nplates=20, dphimax=0.02)
    G = pmx.GSTATE
    tx, ty = np.array(G.FIELDX), np.array(G.FIELDY)
    gw = oracle_gateway()
    it = _interp(gw, seed=11)
    brfs = []
    for k in range(2):
        brfs.append(it.call('fiber', [to_m(fib), 'gps-'], 1)[0])
        it.call('ampliflat', [to_m(GAIN_DB), 'gain'], 0)
    steps = [c['steps'] for c in gw.log if c['cmd'] == 'fiber']
    assert len(steps) == 2 and min(len(x) for x in steps) > 2
    assert not np.array_equal(np.asarray(brfs[0]['theta']), np.asarray(brfs[1]['theta']))
    rx, ry = _m_field(it)
    it.call('dbp', [to_m(fib), 'gps-', _opts(nspan=2, gain=GAIN_DB, steplen=np.concatenate(steps).reshape(1, -1),
                                              spansteps=np.array([[len(x) for x in steps]], dtype=np.float64),
                                              brf=MCell(brfs))], 0)
    ux, uy = _m_field(it)
    assert rel_l2(ux, uy, tx, ty) <= 1e-12
    c = gw.log[-1]
    assert c['fls'][1] == 1 and c['D'][4] == 1
    s = pmx.fiber_setup(fib, 'gps-', rng=np.random.Generator(np.random.PCG64(0)))
    want = dbp_pmd_oracle.dbp_pmd(rx, ry, s.betat, s.db1, s.gam, s.alphalin, 1, s.length, 'no',
                                  [{k: np.asarray(b[k]).ravel() for k in ('db0', 'theta', 'epsilon')} for b in brfs],
                                  nspan=2, gain=10 ** (GAIN_DB / 10), step_len=np.concatenate(steps),
                                  span_steps=[len(x) for x in steps])
    assert rel_l2(ux, uy, *want) <= 1e-13


def test_single_channel():
    """ich = 2, decim = 8 of a 3-channel 'unique' field: the band is [ndfn, 8] with receiver_cohmix's ndfn, and the
    field == dbp_channel_oracle"""
    make_tx(256, 16, nch=3, pavg_mw=4.0)
    fib = base_fiber(slope=0.057, dphimax=0.02)
    G = pmx.GSTATE
    tx, ty = np.array(G.FIELDX), np.array(G.FIELDY)
    s = _setup(fib, 'g-s-')
    from polmux_b200.receiver import channel_ndfn
    for ich in (1, 2):
        m = channel_ndfn(ich)
        want = dco.dbp_channel(tx, ty, s.betat, s.gam, s.alphalin, s.length, 'no', m, 8, nspan=2,
                               gain=10 ** (GAIN_DB / 10), steps_per_span=2)
        gw = oracle_gateway()
        it = _interp(gw)
        it.call('dbp', [to_m(fib), 'g-s-', _opts(nspan=2, gain=GAIN_DB, steps=2, ich=float(ich), decim=8.0)], 0)
        assert list(gw.log[-1]['band']) == [m, 8]
        assert rel_l2(*_m_field(it), *want) <= 1e-13
    assert channel_ndfn(1) != 0


def _python_error(fn):
    with pytest.raises(Exception) as e:
        fn()
    return str(e.value)


@pytest.mark.parametrize('case', ['brf_without_p', 'plate_count', 'brf_count', 'ich_without_decim', 'decim_without_ich',
                                  'no_such_channel', 'multi_column', 'xpm_two_pol', 'wrong_flag'])
def test_errors_are_the_python_mirrors(case):
    """every refusal of dbp.m is an MError with pmx.dbp's message for the same request"""
    if case in ('multi_column', 'xpm_two_pol'):
        make_tx(256, 16, nch=3, ftype='sepfields')
    elif case in ('ich_without_decim', 'decim_without_ich', 'no_such_channel'):
        make_tx(256, 16, nch=3)
    else:
        make_tx(256, 16)
    fib = base_fiber(dgd=0.5, nplates=20)
    b20 = {'db0': np.zeros(20), 'theta': np.zeros(20), 'epsilon': np.zeros(20)}
    b10 = {'db0': np.zeros(10), 'theta': np.zeros(10), 'epsilon': np.zeros(10)}
    flag, py, m = {
        'brf_without_p': ('g-s-', dict(brf=b20), dict(brf=_brf_m(b20))),
        'plate_count': ('gps-', dict(brf=b10), dict(brf=_brf_m(b10))),
        'brf_count': ('gps-', dict(nspan=2, brf=[b20] * 3), dict(nspan=2.0, brf=MCell([_brf_m(b20)] * 3))),
        'ich_without_decim': ('g-s-', dict(ich=2), dict(ich=2.0)),
        'decim_without_ich': ('g-s-', dict(decim=8), dict(decim=8.0)),
        'no_such_channel': ('g-s-', dict(ich=4, decim=8), dict(ich=4.0, decim=8.0)),
        'multi_column': ('g-s-', dict(ich=2, decim=8), dict(ich=2.0, decim=8.0)),
        'xpm_two_pol': ('g-sx', {}, {}),
        'wrong_flag': ('g-s', {}, {}),
    }[case]
    if case == 'multi_column' or case == 'xpm_two_pol':
        fib = base_fiber()
    want = _python_error(lambda: pmx.dbp(fib, flag, **py))
    it = _interp(oracle_gateway())
    before = _m_field(it)
    with pytest.raises(MError) as e:
        it.call('dbp', [to_m(fib), flag, _opts(**m)], 0)
    assert str(e.value) == want
    after = _m_field(it)
    assert np.array_equal(before[0], after[0]) and np.array_equal(before[1], after[1])


def test_fiber_front_end_and_the_shared_set_up_agree_with_python():
    """fiber_setup.m (shared by fiber.m and dbp.m) passes the gateway the scalars pmx.dbp's FiberSetup holds, bit for bit"""
    make_tx(256, 16, nch=3, ftype='sepfields')
    fib = base_fiber(slope=0.057, dphimax=0.02)
    gw = oracle_gateway()
    it = _interp(gw)
    it.call('dbp', [to_m(fib), 'g-s-', _opts(steps=2.0)], 0)
    c = gw.log[-1]
    s = _setup(fib, 'g-s-')
    np.testing.assert_array_equal(c['gam'], s.gam)
    np.testing.assert_array_equal(c['P'], [s.dzmaxt, s.dphimaxt, s.alphalin, s.length, s.nplates, 0])
    sc = s.scalars
    np.testing.assert_array_equal(c['scal'], np.concatenate([[sc['symbolrate'], sc['nsymb'], sc['nt'], sc['b30'],
                                                              sc['dgdrms']], sc['beta1'], sc['beta2']]))


# ---------------------------------------------------------------------------------------------------------------- GPU
def _device_pair(fib, flag, m_opts, py_kw, pmxopt=None, precision=None):
    """-> (field of dbp.m through the compiled gateway, field of pmx.dbp) from the product's current GSTATE"""
    G = pmx.GSTATE
    tx = np.array(G.FIELDX)
    ty = np.array(G.FIELDY) if G.has_y() else None
    it = _interp(mex_bridge.real_gateway(), pmxopt=pmxopt)
    it.call('dbp', [to_m(fib), flag, _opts(**m_opts)], 0)
    mx, my = _m_field(it)
    G.FIELDX = tx
    G.FIELDY = ty if ty is not None else np.zeros((0, 0))
    pmx.dbp(fib, flag, precision=precision, **py_kw)
    return (mx, my), (np.array(G.FIELDX), np.array(G.FIELDY) if G.has_y() else np.zeros((0, 0)))


def _err(m, p):
    if p[1].size:
        return rel_l2(m[0], m[1], p[0], p[1])
    assert m[1].size == 0
    return _rel(m[0], p[0])


ROUTES = {
    'three_pass_2e14': lambda: (make_tx(1024, 16, pavg_mw=4.0), base_fiber(dgd=0.5, nplates=20, manakov='yes'), 'gps-'),
    'onchip_2e10': lambda: (make_tx(64, 16, pavg_mw=4.0), base_fiber(), 'g-s-'),
    'scalar_xpm_2e11x5': lambda: (scalar_tx(64, 32, 5), base_fiber(length=5e4), 'g-sx'),
}


@pytest.mark.gpu
@pytest.mark.parametrize('route', list(ROUTES))
def test_device_equals_python(route):
    """dbp.m through the compiled gateway == pmx.dbp on the same field, <= 1e-13 (2 spans, 16 dB, 4 steps per span)"""
    _, fib, flag = ROUTES[route]()
    m, p = _device_pair(fib, flag, dict(nspan=2.0, gain=GAIN_DB, steps=4.0),
                        dict(nspan=2, gain_db=GAIN_DB, steps_per_span=4))
    assert _err(m, p) <= 1e-13


@pytest.mark.gpu
def test_device_pmd_aware_per_span_brf():
    """PMD-aware DBP at 2^14 with another brf for each span: dbp.m == pmx.dbp(brf=[...])"""
    make_tx(1024, 16, pavg_mw=4.0)
    fib = base_fiber(dgd=0.5, nplates=20)
    g = np.random.Generator(np.random.PCG64(4))
    brfs = [{'db0': g.random(20) * 2 * np.pi - np.pi, 'theta': g.random(20) * np.pi - 0.5 * np.pi,
             'epsilon': 0.5 * np.arcsin(g.random(20) * 2 - 1)} for _ in range(2)]
    m, p = _device_pair(fib, 'gps-', dict(nspan=2.0, gain=GAIN_DB, steps=4.0, brf=MCell([_brf_m(b) for b in brfs])),
                        dict(nspan=2, gain_db=GAIN_DB, steps_per_span=4, brf=brfs))
    assert _err(m, p) <= 1e-13


@pytest.mark.gpu
def test_device_single_channel():
    """single-channel DBP at 2^14, decim 8 (the on-chip route at M = 2^11): dbp.m == pmx.dbp(ich=2, decim=8)"""
    make_tx(1024, 16, nch=3, pavg_mw=4.0)
    fib = base_fiber(slope=0.057, dphimax=0.02)
    m, p = _device_pair(fib, 'g-s-', dict(nspan=2.0, gain=GAIN_DB, steps=4.0, ich=2.0, decim=8.0),
                        dict(nspan=2, gain_db=GAIN_DB, steps_per_span=4, ich=2, decim=8))
    assert _err(m, p) <= 1e-13


@pytest.mark.gpu
def test_device_fp32():
    """PMXOPT.precision = 'f32': dbp.m == pmx.dbp(precision='f32') and within 1e-5 of the FP64 result"""
    make_tx(1024, 16, pavg_mw=4.0)
    fib = base_fiber()
    G = pmx.GSTATE
    tx, ty = np.array(G.FIELDX), np.array(G.FIELDY)
    opts = (dict(nspan=2.0, gain=GAIN_DB, steps=4.0), dict(nspan=2, gain_db=GAIN_DB, steps_per_span=4))
    m32, p32 = _device_pair(fib, 'g-s-', *opts, pmxopt={'precision': 'f32'}, precision='f32')
    G.FIELDX, G.FIELDY = tx, ty
    m64, _ = _device_pair(fib, 'g-s-', *opts)
    assert _err(m32, p32) <= 1e-13
    err = rel_l2(m32[0], m32[1], m64[0], m64[1])
    assert 1e-10 < err < 1e-5, err


@pytest.mark.gpu
def test_device_resident_flow_and_exact_inverse():
    """fiber.m; ampliflat.m x 2 spans, then dbp.m, all resident: the dbp call is a resident hit without an upload, and
    the field equals the same script with PMXOPT.resident = false bit for bit.  With xi = 1 and the steps of
    pmx.fiber(..., trace=True) on the same field, dbp.m returns the Tx field (<= 1e-11)."""
    make_tx(1024, 16, pavg_mw=4.0)
    fib = base_fiber(dphimax=0.02)
    G = pmx.GSTATE
    tx, ty = np.array(G.FIELDX), np.array(G.FIELDY)
    steps = []
    for k in range(2):                                   # the forward steps, from the Python mirror on the same field
        pmx.fiber(fib, 'g-s-', trace=True)
        steps.append(np.asarray(pmx.FIBER_LAST['trace_dz'], dtype=np.float64))
        pmx.ampliflat(GAIN_DB, 'gain')
    assert min(len(x) for x in steps) > 2
    o = _opts(nspan=2.0, gain=GAIN_DB, steplen=np.concatenate(steps).reshape(1, -1),
              spansteps=np.array([[len(x) for x in steps]], dtype=np.float64))
    outs = {}
    for resident in (1.0, 0.0):
        G.FIELDX, G.FIELDY = tx, ty
        gw = mex_bridge.real_gateway()
        it = _interp(gw, pmxopt={'resident': resident})
        for k in range(2):
            it.call('fiber', [to_m(fib), 'g-s-'], 0)
            it.call('ampliflat', [to_m(GAIN_DB), 'gain'], 0)
        s0 = gw.stats()
        it.call('dbp', [to_m(fib), 'g-s-', o], 0)
        s1 = gw.stats()
        up, down, hits = (s1[k] - s0[k] for k in ('uploads', 'downloads', 'resident_hits'))
        assert (up, down, hits) == ((0, 1, 1) if resident else (1, 1, 0))
        outs[resident] = _m_field(it)
    assert np.array_equal(outs[1.0][0], outs[0.0][0]) and np.array_equal(outs[1.0][1], outs[0.0][1])
    err = rel_l2(outs[1.0][0], outs[1.0][1], tx, ty)
    assert err <= 1e-11, err
