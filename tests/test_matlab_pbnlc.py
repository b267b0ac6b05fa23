"""matlab/pbnlc.m -- the M front-end of perturbation-based nonlinearity compensation -- and the gateway command
ssfm_mex('pbnlc', ...), executed by the mini M interpreter (oracle/mini_m).

CPU: pbnlc.m with a gateway whose 'pbnlc' command is served by the numpy table (pbnlc.pb_coefficients) and the stage
oracles (tests/pbnlc_oracle.py, tests/pbnlc_channel_oracle.py) equals those oracles run on the parameters pmx.pbnlc
derives from the same GSTATE; the arguments it sends the gateway are pmx.pbnlc's; every refusal carries pmx.pbnlc's
message.  GPU: the same front-end with the compiled gateway (mexFunction of mex/ssfm_mex.c through the mex.h stand-in)
equals pmx.pbnlc(..., table='device'), keeps the field resident after fiber.m / ampliflat.m, and compensates."""
import importlib
import math
import types

import numpy as np
import pytest

import oracle.fiber_oracle as orc
from oracle.mini_m.interp import MError, to_m
import mex_bridge
import pbnlc_channel_oracle as pco
import pbnlc_oracle as po
import polmux_b200 as pmx
from polmux_b200 import synth
from polmux_b200.receiver import channel_ndfn
from common import base_fiber, make_tx, rel_l2, scalar_tx
from test_matlab_dbp import _interp, _m_field, _opts, _vectors, oracle_gateway as dbp_gateway

pbm = importlib.import_module('polmux_b200.pbnlc')
GAIN_DB = 16.0


def oracle_gateway(log=None):
    """test_matlab_dbp's oracle gateway plus ssfm_mex('pbnlc', ...) served by the oracles: the all-pass step
    (orc.lin_step of the negated dispersion of the whole link), the numpy table, the stage; every call logged"""
    base = dbp_gateway()
    log = [] if log is None else log

    def call(it, a, nargout):
        if a[0] != 'pbnlc':
            return base(it, a, nargout)
        ux, uy, betat, scal, tbetat, L, W, pulse, band, opt = a[1:11]
        L, W = np.asarray(L, np.float64).ravel(), np.asarray(W, np.float64).ravel()
        opt, band = np.asarray(opt, np.float64).ravel(), np.asarray(band, np.float64).ravel()
        pulse, tbetat = np.asarray(pulse, np.float64).ravel(), np.asarray(tbetat, np.float64).ravel()
        log.append(dict(L=L, W=W, opt=opt, band=band, pulse=pulse, tbetat=tbetat, scal=np.asarray(scal).ravel()))
        if opt[0]:
            raise MError('pmx_pb_create: FP64 fields only')
        nfft = np.shape(ux)[0]
        bt = _vectors(scal, nfft, 1, 0)[0][:, 0] if np.size(scal) else np.asarray(betat, np.float64).ravel()
        nspan, lf, alpha, nt, K, nquad, window, prune = L
        nspan, nt, K, nquad, window = int(nspan), int(nt), int(K), int(nquad), int(window)
        ux, uy = np.asarray(ux).ravel(), np.asarray(uy).ravel()
        if opt[2]:
            ux, uy = orc.lin_step(-bt * (lf * nspan), ux), orc.lin_step(-bt * (lf * nspan), uy)
        tab = types.SimpleNamespace(nfft=tbetat.size, betat=tbetat.reshape(-1, 1), length=lf, alphalin=alpha)
        m, n, C = pbm.pb_coefficients(tab, nspan, pulse, K, prune, nt, nquad, window or None)
        if band.size:
            rx, ry, _, _ = pco.pb_channel(ux, uy, pulse, nt, m, n, C, W[:3], W[3], W[5], W[4], int(band[0]), int(band[1]))
        else:
            rx, ry, _, _ = po.stage(ux, uy, pulse, nt, m, n, C, W[:3], W[3], W[5], W[4])
        return [rx.reshape(-1, 1), ry.reshape(-1, 1)][:max(nargout, 1)]
    call.log = log
    return call


def _python_params(fib, flag, nspan, gain_db, xi, K, prune=0.0, nquad=32, window=None, ich=None, decim=None):
    """what pmx.pbnlc derives from the product's GSTATE: (setup, pulse, table setup, nt, weights, gamma, scale, shift)"""
    G = pmx.GSTATE
    f = flag.lower()
    s = pmx.fiber_setup(fib, f[0] + '-' + f[2:])
    s.manakov = f[1] == 'p' and fib.get('manakov', 'no') == 'yes'
    nt, ts, shift = int(G.NT), s, None
    p = synth.cosroll_pulse(nt, 0.2)
    if decim:
        shift = int(channel_ndfn(ich)) if G.NCH > 1 else 0
        p = pbm.channel_pulse(nt, decim, s.nfft)
        ts, nt = pbm.channel_setup(s, shift, decim), nt // decim
    w, gam = pbm.model_weights(s)
    return s, p, ts, nt, w, gam, pbm.scale_factor(s, nspan, gain_db), shift


def _oracle_want(tx, ty, fib, flag, nspan, gain_db, xi, K, **kw):
    s, p, ts, nt, w, gam, scale, shift = _python_params(fib, flag, nspan, gain_db, xi, K, **kw)
    bt = s.betat[:, 0] * (s.length * nspan)
    ux, uy = orc.lin_step(-bt, tx[:, 0]), orc.lin_step(-bt, ty[:, 0])
    m, n, C = pbm.pb_coefficients(ts, nspan, p, K, kw.get('prune', 0.0), nt, kw.get('nquad', 32), kw.get('window'))
    if kw.get('decim'):
        return pco.pb_channel(ux, uy, p, nt, m, n, C, w, gam, scale, xi, shift, kw['decim'])[:2]
    return po.stage(ux, uy, p, nt, m, n, C, w, gam, scale, xi)[:2]


CPU_CASES = {   # make_tx arguments, fiber, flag, m options, python keywords
    'cnlse': ((256, 16), dict(), 'g-s-', dict(nspan=2.0, K=8.0, nquad=8.0), dict(nspan=2, gain_db=None, K=8, nquad=8)),
    'manakov_gain': ((256, 16), dict(manakov='yes'), 'gps-', dict(nspan=3.0, gain=GAIN_DB, K=6.0, nquad=8.0, xi=0.8,
                                                                      prune=1e-3),
                     dict(nspan=3, gain_db=GAIN_DB, K=6, nquad=8, xi=0.8, prune=1e-3)),
    'channel': ((256, 16, 3), dict(slope=0.057), 'g-s-', dict(nspan=2.0, gain=GAIN_DB, K=6.0, nquad=8.0, ich=2.0,
                                                               decim=8.0),
                dict(nspan=2, gain_db=GAIN_DB, K=6, nquad=8, ich=2, decim=8)),
}


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize('case', list(CPU_CASES))
def test_front_end_equals_the_oracle_on_pmx_pbnlcs_parameters(case):
    """pbnlc.m with the oracle-backed 'pbnlc' command == the oracles on pmx.pbnlc's parameters (<= 1e-13), and the
    gateway gets pmx.pbnlc's weights, gamma, scale, link, band exactly and its pulse and table dispersion to 1e-15"""
    tx_args, fkw, flag, mo, pk = CPU_CASES[case]
    make_tx(*tx_args, pavg_mw=4.0)
    fib = base_fiber(**fkw)
    G = pmx.GSTATE
    tx, ty = np.array(G.FIELDX), np.array(G.FIELDY)
    py = dict(pk)
    nspan, gain_db, xi, K = py.pop('nspan'), py.pop('gain_db'), py.pop('xi', 1.0), py.pop('K')
    want = _oracle_want(tx, ty, fib, flag, nspan, gain_db, xi, K, **py)
    gw = oracle_gateway()
    it = _interp(gw)
    it.call('pbnlc', [to_m(fib), flag, _opts(**mo)], 0)
    ux, uy = _m_field(it)
    err = rel_l2(ux[:, 0], uy[:, 0], *want)
    assert err <= 1e-13, err
    s, p, ts, nt, w, gam, scale, shift = _python_params(fib, flag, nspan, gain_db, xi, K, **py)
    c = gw.log[-1]
    np.testing.assert_array_equal(c['W'], [*w, gam, xi, scale])
    np.testing.assert_array_equal(c['L'], [nspan, s.length, s.alphalin, nt, K, py.get('nquad', 32), 0, py.get('prune', 0)])
    np.testing.assert_array_equal(c['band'], [shift, py['decim']] if 'decim' in py else [])
    np.testing.assert_array_equal(c['opt'], [0, 1, 1])
    assert c['pulse'].shape == p.shape and np.abs(c['pulse'] - p).max() <= 1e-15 * np.abs(p).max()
    tb = np.asarray(ts.betat, np.float64)[:, 0]
    assert np.abs(c['tbetat'] - tb).max() <= 1e-15 * np.abs(tb).max()


def test_m_restatements_equal_the_python_functions():
    """the cosroll pulse, channel_setup's dispersion and channel_pulse as pbnlc.m restates them, for several nt / decim"""
    for nsymb, nt, nch, r in ((64, 16, 1, None), (64, 8, 1, None), (256, 16, 3, 8), (128, 32, 3, 4), (256, 16, 3, 2)):
        make_tx(nsymb, nt, nch=nch)
        fib = base_fiber(slope=0.057)
        gw = oracle_gateway()
        it = _interp(gw)
        o = dict(K=0.0, nquad=1.0, xi=0.0) if r is None else dict(K=0.0, nquad=1.0, xi=0.0, ich=3.0, decim=float(r))
        it.call('pbnlc', [to_m(fib), 'g-s-', _opts(**o)], 0)
        c = gw.log[-1]
        s = pmx.fiber_setup(fib, 'g-s-')
        if r is None:
            p = synth.cosroll_pulse(nt, 0.2)
            assert np.array_equal(c['pulse'], p)
        else:
            p = pbm.channel_pulse(nt, r, s.nfft)
            tb = np.asarray(pbm.channel_setup(s, channel_ndfn(3), r).betat, np.float64)[:, 0]
            assert np.abs(c['pulse'] - p).max() <= 1e-15 * np.abs(p).max(), (nt, r)
            assert np.abs(c['tbetat'] - tb).max() <= 1e-15 * np.abs(tb).max(), (nt, r)


def _python_error(fn):
    with pytest.raises(Exception) as e:
        fn()
    return str(e.value)


ERROR_CASES = {   # make_tx call, flag, python keywords, m options
    'ich_without_decim': (lambda: make_tx(256, 16, nch=3), 'g-s-', dict(ich=2), dict(ich=2.0)),
    'decim_without_ich': (lambda: make_tx(256, 16, nch=3), 'g-s-', dict(decim=8), dict(decim=8.0)),
    'no_such_channel': (lambda: make_tx(256, 16, nch=3), 'g-s-', dict(ich=4, decim=8), dict(ich=4.0, decim=8.0)),
    'multiplex_without_decim': (lambda: make_tx(256, 16, nch=3), 'g-s-', {}, {}),
    'multi_column': (lambda: make_tx(256, 16, nch=3, ftype='sepfields'), 'g-s-', dict(ich=2, decim=8),
                     dict(ich=2.0, decim=8.0)),
    'decim_not_pow2': (lambda: make_tx(256, 16, nch=3), 'g-s-', dict(ich=2, decim=3), dict(ich=2.0, decim=3.0)),
    'decim_not_dividing_nt': (lambda: make_tx(256, 8, nch=3), 'g-s-', dict(ich=2, decim=16), dict(ich=2.0, decim=16.0)),
    'no_fieldy': (lambda: scalar_tx(64, 16, 1), 'g-s-', {}, {}),
    'nspan': (lambda: make_tx(64, 16), 'g-s-', dict(nspan=0), dict(nspan=0.0)),
    'K': (lambda: make_tx(64, 16), 'g-s-', dict(K=200), dict(K=200.0)),
    'wrong_flag': (lambda: make_tx(64, 16), 'g-s', {}, {}),
}


@pytest.mark.parametrize('case', list(ERROR_CASES))
def test_errors_are_the_python_mirrors(case):
    """every refusal of pbnlc.m is an MError with pmx.pbnlc's message, and the field is left as it was"""
    mk, flag, py, m = ERROR_CASES[case]
    mk()
    fib = base_fiber()
    want = _python_error(lambda: pmx.pbnlc(fib, flag, **py))
    it = _interp(oracle_gateway())
    before = _m_field(it)
    with pytest.raises(MError) as e:
        it.call('pbnlc', [to_m(fib), flag, _opts(**m)], 0)
    assert str(e.value) == want
    after = _m_field(it)
    assert np.array_equal(before[0], after[0]) and np.array_equal(before[1], after[1])


def test_fp32_is_refused():
    make_tx(64, 16)
    it = _interp(oracle_gateway(), pmxopt={'precision': 'f32'})
    with pytest.raises(MError, match='pmx_pb_create: FP64 fields only'):
        it.call('pbnlc', [to_m(base_fiber()), 'g-s-', _opts()], 0)


# ---------------------------------------------------------------------------------------------------------------- GPU
def _device_pair(fib, flag, m_opts, py_kw, pmxopt=None):
    """-> (field of pbnlc.m through the compiled gateway, field of pmx.pbnlc(table='device')) from the current GSTATE"""
    G = pmx.GSTATE
    tx, ty = np.array(G.FIELDX), np.array(G.FIELDY)
    it = _interp(mex_bridge.real_gateway(), pmxopt=pmxopt)
    it.call('pbnlc', [to_m(fib), flag, _opts(**m_opts)], 0)
    mx, my = _m_field(it)
    G.FIELDX, G.FIELDY = tx, ty
    pmx.pbnlc(fib, flag, table='device', **py_kw)
    return (mx, my), (np.array(G.FIELDX), np.array(G.FIELDY))


GPU_ROUTES = {
    'natural_2e10': (lambda: make_tx(64, 16, pavg_mw=4.0), dict(), 'g-s-', dict(), {}),
    'transposed_2e14': (lambda: make_tx(1024, 16, pavg_mw=4.0), dict(manakov='yes'), 'gps-', dict(), {}),
    'channel_2e14': (lambda: make_tx(1024, 16, nch=3, pavg_mw=4.0), dict(slope=0.057), 'g-s-', dict(ich=2.0, decim=8.0),
                     dict(ich=2, decim=8)),
}


@pytest.mark.gpu
@pytest.mark.parametrize('route', list(GPU_ROUTES))
def test_device_equals_python(route):
    """pbnlc.m through the compiled gateway == pmx.pbnlc(table='device') on the same field, <= 1e-13 (3 spans, 16 dB,
    K = 16)"""
    mk, fkw, flag, mo, pk = GPU_ROUTES[route]
    mk()
    m, p = _device_pair(base_fiber(**fkw), flag, dict(nspan=3.0, gain=GAIN_DB, K=16.0, **mo),
                        dict(nspan=3, gain_db=GAIN_DB, K=16, **pk))
    err = rel_l2(m[0], m[1], p[0], p[1])
    print('pbnlc.m vs pmx.pbnlc (%s): rel_l2 %.2e' % (route, err))
    assert err <= 1e-13


@pytest.mark.gpu
def test_device_resident_flow():
    """fiber.m; ampliflat.m x 2 spans, then pbnlc.m, all resident: the pbnlc call is a resident hit without an upload,
    and the field equals the same script with PMXOPT.resident = false bit for bit"""
    make_tx(1024, 16, pavg_mw=4.0)
    fib = base_fiber(dphimax=0.02)
    G = pmx.GSTATE
    tx, ty = np.array(G.FIELDX), np.array(G.FIELDY)
    outs = {}
    for resident in (1.0, 0.0):
        G.FIELDX, G.FIELDY = tx, ty
        gw = mex_bridge.real_gateway()
        it = _interp(gw, pmxopt={'resident': resident})
        for k in range(2):
            it.call('fiber', [to_m(fib), 'g-s-'], 0)
            it.call('ampliflat', [to_m(GAIN_DB), 'gain'], 0)
        s0 = gw.stats()
        it.call('pbnlc', [to_m(fib), 'g-s-', _opts(nspan=2.0, gain=GAIN_DB, K=16.0)], 0)
        s1 = gw.stats()
        up, down, hits = (s1[k] - s0[k] for k in ('uploads', 'downloads', 'resident_hits'))
        assert (up, down, hits) == ((0, 1, 1) if resident else (1, 1, 0))
        outs[resident] = _m_field(it)
    assert np.array_equal(outs[1.0][0], outs[0.0][0]) and np.array_equal(outs[1.0][1], outs[0.0][1])


@pytest.mark.gpu
def test_gateway_pbnlc_lowers_the_residual_below_cd_only():
    """one channel, 5 x 80 km at 4 mW, noise-free (test_pbnlc's link): through pbnlc.m and the compiled gateway the
    symbol-centre residual after PB-NLC (K = 48) is below that of the all-pass step alone (xi = 0)"""
    tp = importlib.import_module('test_pbnlc')
    nsymb, nt, nspan = 1024, 8, 5
    tx, rx, s = tp._link(nsymb, nt, 4.0, nspan, False)
    gain_db = 10 * math.log10(math.exp(s.alphalin * s.length))
    fib = base_fiber(dphimax=1e-3)
    G = pmx.GSTATE
    res = {}
    for what, o in (('cd', dict(xi=0.0, K=0.0)), ('pbnlc', dict(xi=1.0, K=48.0))):
        bt = s.betat * (s.length * nspan)
        G.FIELDX, G.FIELDY = orc.lin_step(bt, rx[0]), orc.lin_step(bt, rx[1])
        it = _interp(mex_bridge.real_gateway())
        it.call('pbnlc', [to_m(fib), 'g-s-', _opts(nspan=float(nspan), gain=gain_db, **o)], 0)
        mx, my = _m_field(it)
        G.FIELDX, G.FIELDY = mx, my
        res[what] = tp._symbol_residual(G, tx, 1.0, nt)
    print('pbnlc.m symbol-centre residual vs Tx: CD only %.4f, PB-NLC (K=48) %.4f' % (res['cd'], res['pbnlc']))
    assert res['pbnlc'] < 0.8 * res['cd']
