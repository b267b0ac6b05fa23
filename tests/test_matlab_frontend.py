"""matlab/fiber.m and matlab/ampliflat.m -- the thin M front-ends that replace the toolbox's fiber.m on the path --
executed by the mini M interpreter (oracle/mini_m).

CPU: the front-end with an oracle-backed ssfm_mex reproduces the goldens the interpreted ORIGINAL fiber.m produced
(same plate draws from the same rand stream, same DELAY / DISP, same brf, same simul_out text), starting from the Tx
field the interpreted reset_all.m / create_field.m left in GSTATE (stored with each golden).  The toolbox functions the
front-ends call (avg_power.m, myfilter.m, fastexp.m) are stood in for by the oracle's restatements, pinned on the
interpreted originals by test_golden and test_receiver_oracle.  Where the toolbox's own M source is at hand, the
scripts' calls also run unchanged with matlab/ first on the path against it.
GPU: the same front-end with the real gateway (mexFunction of mex/ssfm_mex.c through the mex.h stand-in) against the
goldens, including C1 at its full size, the resident span loop fiber(); ampliflat(); and the FP32 option."""
import glob
import json
import os

import numpy as np
import pytest

import oracle.fiber_oracle as orc
from oracle.mini_m.interp import Interp, MStruct, MError, from_m, to_m
from polmux_b200 import synth
import mex_bridge

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, 'tests', 'golden')
MDIR = os.path.join(ROOT, 'matlab')
REF = '/root/reference'
CASES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLD, '*.npz')))
needs_ref = pytest.mark.skipif(not os.path.exists(os.path.join(REF, 'create_field.m')), reason='reference tree not present')


def load(name):
    z = np.load(os.path.join(GOLD, name + '.npz'))
    return z, json.loads(str(z['meta']))


def globals_from_python(it, nsymb, nt, nch, rate, pavg, fx, fy, lams=None):
    """GSTATE / CONSTANTS as reset_all.m + create_field.m leave them (for runs without the reference tree)."""
    n = nsymb * nt
    it.globals['CONSTANTS'] = MStruct({'CLIGHT': to_m(orc.CLIGHT), 'HPLANCK': to_m(orc.HPLANCK),
                                       'ECHARGE': to_m(orc.ECHARGE), 'KBOLTZMANN': to_m(orc.KBOLTZMANN)})
    fn = np.fft.fftshift(-nt / 2.0 + np.arange(n) / nsymb).reshape(1, -1)
    npol = 2 if fy is not None else 1
    it.globals['GSTATE'] = MStruct({
        'NSYMB': to_m(nsymb), 'NT': to_m(nt), 'NCH': to_m(nch), 'FN': fn, 'SYMBOLRATE': to_m(rate),
        'LAMBDA': (synth.wdm_lambdas(nch) if lams is None else lams).reshape(1, -1),
        'POWER': np.full((1, nch), float(pavg)), 'FIELDX': np.array(fx), 'FIELDY': np.zeros((0, 0)) if fy is None else np.array(fy),
        'DELAY': np.zeros((npol, nch)), 'DISP': np.zeros((npol, nch)), 'PRINT': np.array([[False]]), 'DIR': 'sim'})
    it.globals['PMXOPT'] = np.zeros((0, 0))


def tx_from_golden(it, m, z):
    """GSTATE as the interpreted reset_all.m + create_field.m left it: the golden's stored Tx field and power"""
    globals_from_python(it, m['nsymb'], m['nt'], m['nch'], m['rate'], m['pavg'], z['tx_FIELDX'],
                        z['tx_FIELDY'] if m['two_pol'] else None)
    it.globals['GSTATE']['POWER'] = np.array(z['tx_POWER'], dtype=np.float64).reshape(1, -1)


def avg_power_stand_in(m):
    """the toolbox's avg_power.m (called by matlab/ampliflat.m for 'fixpower') as the oracle's restatement, pinned on
    the interpreted avg_power.m by test_golden"""
    def avg_power(it_, a, nargout):
        Gm = it_.globals['GSTATE']
        gs = orc.reset_all(m['nsymb'], m['nt'], m['nch'])
        gs.FIELDX, fy = np.asarray(Gm['FIELDX']), np.asarray(Gm['FIELDY'])
        gs.FIELDY = fy if fy.size else None
        assert a[1] == 'abs'
        return [to_m(orc.avg_power_abs(gs, int(np.asarray(a[0]).ravel()[0])))]
    return avg_power


@pytest.mark.parametrize('scalmode', [0, 1])
@pytest.mark.parametrize('name', CASES)
def test_front_end_reproduces_the_interpreted_original(name, scalmode):
    """matlab/fiber.m + the Tx field of the interpreted create_field.m + an oracle-backed ssfm_mex
    == the interpreted original fiber.m: fields <= 1e-13, DELAY / DISP, the brf struct and its plate draws"""
    z, m = load(name)
    calls = []
    it = Interp([MDIR], rng=np.random.Generator(np.random.PCG64(m['seed'])))
    it.builtins['ssfm_mex'] = mex_bridge.oracle_gateway(calls)
    tx_from_golden(it, m, z)
    it.globals['PMXOPT'] = MStruct({'scalar': to_m(float(scalmode))})
    want_brf = 'brf_theta' in z.files
    res = it.call('fiber', [to_m(m['fiber']), m['flag']], 1 if want_brf else 0)
    G = it.globals['GSTATE']
    if z['out_FIELDY'].size:
        err = orc.rel_l2(G['FIELDX'], G['FIELDY'], z['out_FIELDX'], z['out_FIELDY'])
    else:
        err = float(np.linalg.norm(G['FIELDX'] - z['out_FIELDX']) / np.linalg.norm(z['out_FIELDX']))
        assert np.size(G['FIELDY']) == 0
    assert err < 1e-13, err
    np.testing.assert_allclose(G['DELAY'], z['out_DELAY'], rtol=1e-13, atol=1e-13)
    np.testing.assert_allclose(G['DISP'], z['out_DISP'], rtol=1e-13, atol=1e-13)
    assert len(calls) == 1 and calls[0]['scalar_field'] == (0.0 if m['two_pol'] or m['fiber'].get('dgd') else 1.0)
    if want_brf:
        brf = from_m(res[0])
        for k in ('db0', 'theta', 'epsilon'):
            np.testing.assert_array_equal(np.asarray(brf[k]).ravel(), z['brf_' + k])
        np.testing.assert_allclose(np.asarray(brf['betat']), z['brf_betat'], rtol=1e-15, atol=0)
        np.testing.assert_allclose(np.asarray(brf['db1']), z['brf_db1'], rtol=1e-15, atol=0)
        assert float(np.asarray(brf['lcorr']).ravel()[0]) == float(z['brf_lcorr'][0])
    if 'amp_FIELDX' in z.files:    # matlab/ampliflat.m ('gain' and 'fixpower', the latter through the toolbox's avg_power.m)
        a = m['amp']
        it.builtins['avg_power'] = avg_power_stand_in(m)
        opt = MStruct({'f': to_m(a['f']), 'noise': to_m(z['amp_noise'])})
        it.call('ampliflat', [to_m(a['gain']), a.get('atype', 'gain'), opt], 0)
        G = it.globals['GSTATE']
        assert orc.rel_l2(G['FIELDX'], G['FIELDY'], z['amp_FIELDX'], z['amp_FIELDY']) < 1e-13


@pytest.mark.parametrize('name', sorted(os.path.basename(p)[len('simul_out_'):-5] for p in
                                        glob.glob(os.path.join(GOLD, 'simul_out_*.json'))))
def test_front_end_prints_the_same_summary(name):
    """GSTATE.PRINT: the block matlab/fiber.m appends to simul_out is character-identical to the original's (Tx field
    from the oracle's create_field, pinned on the interpreted create_field.m by test_golden)"""
    m = json.load(open(os.path.join(GOLD, 'simul_out_%s.json' % name)))
    ex, ey, _, _ = synth.pdm_qpsk(m['nsymb'], m['nt'], m['nch'])
    gs = orc.reset_all(m['nsymb'], m['nt'], m['nch'])
    gs.SYMBOLRATE, gs.POWER, gs.LAMBDA = m['rate'], np.full(m['nch'], float(m['pavg'])), synth.wdm_lambdas(m['nch'])
    orc.create_field(gs, m['ftype'], ex, ey if m['two_pol'] else None, power_average=True)
    it = Interp([MDIR], rng=np.random.Generator(np.random.PCG64(m['seed'])))
    it.builtins['ssfm_mex'] = mex_bridge.oracle_gateway()
    tx_from_golden(it, m, {'tx_FIELDX': gs.FIELDX, 'tx_FIELDY': gs.FIELDY, 'tx_POWER': gs.POWER})
    G = it.globals['GSTATE'].copy()
    G['PRINT'] = to_m(True)
    G['DIR'] = 'sim'
    it.globals['GSTATE'] = G
    it.printed = []
    it.call('fiber', [to_m(m['fiber']), m['flag']], 0)
    assert ''.join(it.printed) == m['text']


def test_front_end_errors_like_the_original():
    it = Interp([MDIR])
    it.builtins['ssfm_mex'] = mex_bridge.oracle_gateway()
    z, m = load('scalar_gs')
    tx_from_golden(it, m, z)
    with pytest.raises(MError, match='wrong flag'):
        it.call('fiber', [to_m(m['fiber']), 'abcd'], 0)
    with pytest.raises(MError, match='only for channels separated'):
        it.call('fiber', [to_m(m['fiber']), 'g--x'], 0)
    with pytest.raises(MError, match='Missing DGD'):
        it.call('fiber', [to_m(m['fiber']), 'gps-'], 0)
    with pytest.raises(MError, match='wrong string atype'):
        it.call('ampliflat', [to_m(3.0), 'boost'], 0)
    z3, m3 = load('wdm3_unique_manakov')         # three channels in one 'unique' field
    tx_from_golden(it, m3, z3)
    with pytest.raises(MError, match='only for channels separated'):
        it.call('ampliflat', [to_m(1.0), 'fixpower'], 0)
    tx_from_golden(it, m, z)
    z, m = load('cnlse_nopmd')
    tx_from_golden(it, m, z)
    with pytest.raises(MError, match='absence of polarization'):
        it.call('fiber', [to_m(dict(m['fiber'], ltol=1e-6)), 'g-s-'], 0)


@needs_ref
@pytest.mark.parametrize('script', ['Run_my_PDM_QPSK', 'ex24_pmd', 'ex06_ber'])
def test_script_call_sequences_run_unchanged(script):
    """The in-line device calls of the reference's scripts, verbatim, with matlab/ first on the path against the toolbox
    alone: Run_my_PDM_QPSK.m:117-122 (create_field('sepfields',...); fiber(fib,'g---')), ex24_pmd.m:78-100 (a PMF given by
    scalar db0/theta/epsilon: fiber(tx,'gp--'); ampliflat(Gerbio,'gain')) and the span loop of ex06_ber.m:110-115
    (fiber(tx,'g-sx'); fiber(comp,'g-sx'); ampliflat(Gerbio,'gain',ampli) with injected noise)"""
    out = {}
    for path in ([REF], [MDIR, REF]):
        it = Interp(path, rng=np.random.Generator(np.random.PCG64(3)))
        if len(path) == 2:
            it.builtins['ssfm_mex'] = mex_bridge.oracle_gateway()
        it.globals['PMXOPT'] = np.zeros((0, 0))
        if script == 'Run_my_PDM_QPSK':
            nsymb, nt, nch = 64, 16, 1
            ex, ey, _, _ = synth.pdm_qpsk(nsymb, nt, nch)
            fib = dict(length=1e3, alphadB=0.2, aeff=80.0, n2=2.7e-20, **{'lambda': 1550.0}, disp=17.0, slope=0.0, dphimax=5e-3,
                       dzmax=2e4, dgd=1.0, nplates=10.0, manakov='no')
            calls = [('create_field', ['sepfields', to_m(ex), to_m(ey), MStruct({'power': 'average'})]),
                     ('fiber', [to_m(fib), 'g---'])]
        elif script == 'ex24_pmd':
            nsymb, nt, nch = 32, 32, 1
            ex, _, _, _ = synth.pdm_qpsk(nsymb, nt, nch)
            tx = dict(length=1e5, alphadB=0.2, aeff=80.0, n2=2.7e-20, **{'lambda': 1550.0}, disp=17.0, slope=0.0, dphimax=5e-3,
                      dzmax=2e4, db0=0.0, theta=np.pi / 4, epsilon=np.pi / 4, dgd=0.5, nplates=20.0)
            calls = [('create_field', ['unique', to_m(ex), to_m(np.zeros_like(ex))]),
                     ('fiber', [to_m(tx), 'gp--']), ('ampliflat', [to_m(20.0), 'gain'])]
        else:
            nsymb, nt, nch = 32, 32, 1
            ex, _, _, _ = synth.pdm_qpsk(nsymb, nt, nch)
            tx = dict(length=1e5, alphadB=0.2, aeff=80.0, n2=2.7e-20, **{'lambda': 1550.0}, disp=17.0, slope=0.0, dphimax=3e-3,
                      dzmax=2e4)
            comp = dict(tx, length=1.7e4, alphadB=0.6, aeff=20.0, disp=-100.0)
            g = np.random.Generator(np.random.PCG64(8))
            calls = [('create_field', ['unique', to_m(ex), np.zeros((0, 0)), MStruct({'power': 'average'})])]
            for k in range(2):
                noise = g.standard_normal((nsymb * nt, 2)) + 1j * g.standard_normal((nsymb * nt, 2))
                calls += [('fiber', [to_m(tx), 'g-sx']), ('fiber', [to_m(comp), 'g-sx']),
                          ('ampliflat', [to_m(30.2), 'gain', MStruct({'f': to_m(6.0), 'noise': noise})])]
        it.call('reset_all', [to_m(nsymb), to_m(nt), to_m(nch)], 0)
        G = it.globals['GSTATE'].copy()
        G['SYMBOLRATE'], G['LAMBDA'], G['POWER'] = to_m(10.0), to_m(np.array([[1550.0]])), to_m(np.array([[4.0]]))
        it.globals['GSTATE'] = G
        for name, args in calls:
            it.call(name, args, 0)
        G = it.globals['GSTATE']
        out[len(path)] = (np.array(G['FIELDX']), np.array(G['FIELDY']), np.array(G['DELAY']), np.array(G['DISP']))
    a, b = out[1], out[2]
    assert a[0].shape == b[0].shape and a[1].shape == b[1].shape
    assert np.linalg.norm(a[0] - b[0]) <= 1e-13 * np.linalg.norm(a[0])
    if a[1].size:
        assert np.linalg.norm(a[1] - b[1]) <= 1e-13 * max(np.linalg.norm(a[1]), 1e-300) + 1e-18
    np.testing.assert_allclose(b[2], a[2], rtol=1e-13, atol=1e-13)
    np.testing.assert_allclose(b[3], a[3], rtol=1e-13, atol=1e-13)


# ---- matlab/receiver_cohmix.m
RXGOLD = os.path.join(GOLD, 'rx')
RXCASES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(RXGOLD, 'rx_*.npz')))


def _rx_case(name):
    z = np.load(os.path.join(RXGOLD, name + '.npz'))
    m = json.loads(str(z['meta']))
    x = dict(m['x'])
    if x.get('lophasenoise') == 'PN':
        x['lophasenoise'] = z['lophasenoise'].reshape(-1, 1)
    return z, m, MStruct({k: (v if isinstance(v, str) else to_m(v)) for k, v in x.items()})


def _rx_toolbox_stand_ins(it):
    """myfilter.m / fastexp.m belong to the toolbox: the oracle's restatement (pinned by test_receiver_oracle)"""
    import oracle.receiver_oracle as rxo
    it.builtins['myfilter'] = lambda it_, a, nargout: [rxo.myfilter(a[0], np.asarray(a[1]), float(np.asarray(a[2]).ravel()[0]),
                                                                   float(np.asarray(a[3]).ravel()[0]) if len(a) > 3 else 0).reshape(-1, 1)]
    it.builtins['fastexp'] = lambda it_, a, nargout: [np.cos(np.asarray(a[0])) + 1j * np.sin(np.asarray(a[0]))]


def _rx_globals(it, z, m):
    globals_from_python(it, m['nsymb'], m['nt'], m['nch'], m['rate'], m['pavg'], z['FIELDX'],
                        z['FIELDY'] if z['FIELDY'].size else None)
    G = it.globals['GSTATE']
    G['POWER'] = z['POWER'].reshape(1, -1)
    G['FIELDX_TX'] = np.array(z['FIELDX_TX'])
    G['FIELDY_TX'] = np.array(z['FIELDY_TX']) if z['FIELDY_TX'].size else np.zeros((0, 0))


def _rx_check(it, z, m, x, tol):
    before = np.array(it.globals['GSTATE']['FIELDX'])
    iric, xo = it.call('receiver_cohmix', [to_m(float(m['ich'])), x], 2)
    assert np.shape(iric) == z['Iric'].shape
    assert np.linalg.norm(np.asarray(iric) - z['Iric']) <= tol * np.linalg.norm(z['Iric'])
    assert abs(float(np.asarray(xo['avgebx']).ravel()[0]) / float(z['avgebx'][0]) - 1) < tol
    if z['avgeby'].size:
        assert abs(float(np.asarray(xo['avgeby']).ravel()[0]) / float(z['avgeby'][0]) - 1) < tol
    pd = float(np.asarray(xo['post_delay'], dtype=np.float64).ravel()[0])
    assert abs(pd - float(z['post_delay'][0])) <= 1e-13 * max(1.0, abs(pd))
    assert np.array_equal(np.asarray(it.globals['GSTATE']['FIELDX']), before)      # GSTATE is left unchanged
    one = it.call('receiver_cohmix', [to_m(float(m['ich'])), x], 1)[0]
    assert np.array_equal(np.asarray(one), np.asarray(iric))


@pytest.mark.parametrize('name', RXCASES)
def test_receiver_front_end_reproduces_the_interpreted_original(name):
    """matlab/receiver_cohmix.m + the oracle's myfilter / fastexp + an oracle-backed ssfm_mex
    == the interpreted original receiver_cohmix.m: currents, avgebx / avgeby, post_delay"""
    z, m, x = _rx_case(name)
    it = Interp([MDIR])
    it.builtins['ssfm_mex'] = mex_bridge.oracle_gateway()
    _rx_toolbox_stand_ins(it)
    _rx_globals(it, z, m)
    _rx_check(it, z, m, x, 1e-13)


# ---- matlab/inverse_pmd.m
INVGOLD = os.path.join(GOLD, 'invpmd', 'invpmd_two_fibers.npz')
INVVARIANTS = {'plain': None, 'mat_nogvd': {'mat': 'MAT', 'gvd': 'no'}, 'noapply': {'apply': 'no'}, 'apply_n': {'apply': 'n', 'mat': 'MAT'}}


def _inv_run(it, tag):
    from oracle.mini_m.interp import MCell
    z = np.load(INVGOLD)
    m = json.loads(str(z['meta']))
    globals_from_python(it, m['nsymb'], m['nt'], 1, m['rate'], m['pavg'], z['prop_FIELDX'], z['prop_FIELDY'])
    it.globals['GSTATE']['DISP'] = np.ones((2, 1))
    brfs = MCell([MStruct({k: (to_m(float(z['brf%d_%s' % (f, k)][0])) if k == 'lcorr' else np.array(z['brf%d_%s' % (f, k)], dtype=np.float64).reshape(-1, 1) if k in ('db0', 'theta', 'epsilon') else np.array(z['brf%d_%s' % (f, k)]))
                           for k in ('db0', 'theta', 'epsilon', 'lcorr', 'betat', 'db1')}) for f in range(2)])
    opt = INVVARIANTS[tag]
    args = [brfs] + ([MStruct({k: (to_m(z['mat']) if v == 'MAT' else v) for k, v in opt.items()})] if opt else [])
    uinv, u = it.call('inverse_pmd', args, 2)
    return z, np.asarray(uinv), np.asarray(u), it.globals['GSTATE']


def _inv_check(z, tag, uinv, u, G, tol):
    assert uinv.shape == z[tag + '_Uinv'].shape and u.shape == uinv.shape
    np.testing.assert_allclose(uinv, z[tag + '_Uinv'], rtol=0, atol=tol)
    np.testing.assert_allclose(u, z[tag + '_U'], rtol=0, atol=tol)
    assert orc.rel_l2(G['FIELDX'], G['FIELDY'], z[tag + '_FIELDX'], z[tag + '_FIELDY']) < tol
    applied = tag != 'noapply'
    np.testing.assert_array_equal(np.asarray(G['DISP']), np.zeros((2, 1)) if applied else np.ones((2, 1)))


@pytest.mark.parametrize('tag', list(INVVARIANTS))
def test_inverse_pmd_front_end_reproduces_the_interpreted_original(tag):
    """matlab/inverse_pmd.m + an oracle-backed ssfm_mex('invpmd', ...) == the interpreted original inverse_pmd.m with every option"""
    it = Interp([MDIR])
    it.builtins['ssfm_mex'] = mex_bridge.oracle_gateway()
    z, uinv, u, G = _inv_run(it, tag)
    _inv_check(z, tag, uinv, u, G, 1e-12)


# ------------------------------------------------------------------------------------------------ GPU
def _gpu_interp(seed):
    it = Interp([MDIR], rng=np.random.Generator(np.random.PCG64(seed)))
    gw = mex_bridge.real_gateway()
    it.builtins['ssfm_mex'] = gw
    return it, gw


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['manakov_100plates_80km', 'cnlse_10plates_100km', 'sep3_manakov', 'pmf_single', 'scalar_gs',
                                  'scalar_sep3_gsx', 'scalar_ltol_gs', 'scalar_dphiadapt_sep3_gsx', 'cnlse_nopmd',
                                  'small_ex06_gsx_2e10', 'small_ex10_sep5_gsx_2e11', 'small_2pol_cnlse_2e9',
                                  'fixpower_sep3_manakov', 'fixpower_scalar_sep3_gsx'])
def test_interpreted_front_end_on_the_device(name):
    """matlab/fiber.m interpreted, its ssfm_mex the compiled gateway on the GPU: all three dispatches (matrix_ssfm,
    scalar_ssfm, scalar_a_ssfm) against the interpreted original's goldens, FP64 <= 1e-10"""
    z, m = load(name)
    it, gw = _gpu_interp(m['seed'])
    two = m['two_pol']
    globals_from_python(it, m['nsymb'], m['nt'], m['nch'], m['rate'], m['pavg'], z['tx_FIELDX'],
                        z['tx_FIELDY'] if two else None)
    it.call('fiber', [to_m(m['fiber']), m['flag']], 0)
    G = it.globals['GSTATE']
    if z['out_FIELDY'].size:
        err = orc.rel_l2(G['FIELDX'], G['FIELDY'], z['out_FIELDX'], z['out_FIELDY'])
    else:
        err = float(np.linalg.norm(G['FIELDX'] - z['out_FIELDX']) / np.linalg.norm(z['out_FIELDX']))
    assert err < 1e-10, err
    np.testing.assert_allclose(G['DELAY'], z['out_DELAY'], rtol=1e-13, atol=1e-13)
    np.testing.assert_allclose(G['DISP'], z['out_DISP'], rtol=1e-13, atol=1e-13)
    if 'amp' in m:
        # matlab/ampliflat.m, 'fixpower' included (its avg_power.m call answered by the oracle's restatement)
        it.builtins['avg_power'] = avg_power_stand_in(m)
        opt = MStruct({'f': to_m(m['amp']['f']), 'noise': to_m(z['amp_noise'])})
        it.call('ampliflat', [to_m(m['amp']['gain']), m['amp'].get('atype', 'gain'), opt], 0)
        G = it.globals['GSTATE']
        assert orc.rel_l2(G['FIELDX'], G['FIELDY'], z['amp_FIELDX'], z['amp_FIELDY']) < 1e-10


@pytest.mark.gpu
@pytest.mark.parametrize('name', RXCASES)
def test_interpreted_receiver_front_end_on_the_device(name):
    """matlab/receiver_cohmix.m interpreted, its ssfm_mex('cohmix', ...) the compiled gateway on the GPU (pmx_cohmix_run),
    against the interpreted original's goldens, FP64 <= 1e-10 (myfilter / fastexp as the oracle's restatement)."""
    z, m, x = _rx_case(name)
    it, gw = _gpu_interp(0)
    _rx_toolbox_stand_ins(it)
    _rx_globals(it, z, m)
    _rx_check(it, z, m, x, 1e-10)


@pytest.mark.gpu
@pytest.mark.parametrize('tag', list(INVVARIANTS))
def test_interpreted_inverse_pmd_front_end_on_the_device(tag):
    """matlab/inverse_pmd.m interpreted, its ssfm_mex('invpmd', ...) the compiled gateway on the GPU (pmx_inverse_pmd_run)"""
    it, gw = _gpu_interp(0)
    z, uinv, u, G = _inv_run(it, tag)
    _inv_check(z, tag, uinv, u, G, 1e-10)


@pytest.mark.gpu
def test_interpreted_front_end_c1_full_size_and_resident_span_loop():
    """C1 at its full size through the interpreted front-end against the interpreted original; then the script loop
    `fiber(x,flag); ampliflat(G,'gain',opt);` three times: the field is uploaded once (the gateway keeps it in HBM and
    recognises the arrays it handed back), every call still returns its arrays to the interpreter, and the result
    equals the same loop with PMXOPT.resident = false bit for bit; FP32 option within 1e-5 (Manakov golden)"""
    import polmux_b200 as pmx
    z = np.load(os.path.join(GOLD, 'big', 'c1_cnlse_10plates_100km_2e16.npz'))
    m = json.loads(str(z['meta']))
    ex, ey, _, _ = synth.pdm_qpsk(m['nsymb'], m['nt'], 1)
    pmx.reset_all(m['nsymb'], m['nt'], 1)
    P = pmx.GSTATE
    P.SYMBOLRATE, P.POWER, P.LAMBDA = m['rate'], np.array([float(m['pavg'])]), synth.wdm_lambdas(1)
    pmx.create_field('unique', ex, ey, {'power': 'average'})
    tx_x, tx_y = np.array(P.FIELDX), np.array(P.FIELDY)
    it, gw = _gpu_interp(m['seed'])
    globals_from_python(it, m['nsymb'], m['nt'], 1, m['rate'], m['pavg'], tx_x, tx_y)
    it.call('fiber', [to_m(m['fiber']), 'gps-'], 0)
    G = it.globals['GSTATE']
    assert orc.rel_l2(G['FIELDX'], G['FIELDY'], z['out_FIELDX'], z['out_FIELDY']) < 1e-10
    # span loop, resident and per-call
    fib = dict(m['fiber'], length=2e4)
    outs = {}
    for resident in (1.0, 0.0):
        it, gw = _gpu_interp(5)
        globals_from_python(it, m['nsymb'], m['nt'], 1, m['rate'], m['pavg'], tx_x, tx_y)
        it.globals['PMXOPT'] = MStruct({'resident': to_m(resident)})
        s0 = gw.stats()
        for k in range(3):
            it.call('fiber', [to_m(fib), 'gps-'], 0)
            it.call('ampliflat', [to_m(4.0), 'gain', MStruct({'f': to_m(5.0)})], 0)
        s1 = gw.stats()
        G = it.globals['GSTATE']
        outs[resident] = (np.array(G['FIELDX']), np.array(G['FIELDY']))
        up, down, hits = (s1[k] - s0[k] for k in ('uploads', 'downloads', 'resident_hits'))
        assert down == 6
        assert (up, hits) == ((1, 5) if resident else (6, 0))
    assert np.array_equal(outs[1.0][0], outs[0.0][0]) and np.array_equal(outs[1.0][1], outs[0.0][1])
    # FP32 option of the front-end (PMXOPT.precision = 'f32'), on the Manakov golden: within the mode's 1e-5
    z, m = load('manakov_100plates_80km')
    it, gw = _gpu_interp(m['seed'])
    globals_from_python(it, m['nsymb'], m['nt'], 1, m['rate'], m['pavg'], z['tx_FIELDX'], z['tx_FIELDY'])
    it.globals['PMXOPT'] = MStruct({'precision': 'f32'})
    it.call('fiber', [to_m(m['fiber']), m['flag']], 0)
    G = it.globals['GSTATE']
    err = orc.rel_l2(G['FIELDX'], G['FIELDY'], z['out_FIELDX'], z['out_FIELDY'])
    assert 1e-9 < err < 1e-5, err
