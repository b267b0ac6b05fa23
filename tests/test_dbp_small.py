"""Digital backpropagation of small fields and of the scalar path (pmx_dbp_create / pmx_dbp_exec on the single-launch
on-chip kernel, pmx_onchip.cuh with DBP = true): two-polarization fields of 2^6 to 2^11 samples, PMD-blind and PMD-aware,
and the scalar path from 2^6 to 2^12 samples with and without cross-phase modulation ('x': the nonlinear step of every
column sees the power of all backpropagated columns).  The sizes are those of the reference's small scripts, ex06_ber.m
(32 x 32, one channel, 'g-sx') and ex10_wdm.m (64 x 32, five separate channels, 'g-sx').

Oracles: tests/dbp_oracle.py and tests/dbp_pmd_oracle.py for two polarizations, tests/dbp_scalar_oracle.py for the scalar
path; the latter is tied to the pinned forward oracle by its exact inverse of scalar_ssfm."""
import ctypes
import math

import numpy as np
import pytest

import oracle.fiber_oracle as orc
import dbp_oracle
import dbp_pmd_oracle as dpo
import dbp_scalar_oracle as dso
import polmux_b200 as pmx
from polmux_b200 import _lib, mc
from polmux_b200.dbp import dbp_plan
from polmux_b200.fiber import fiber_setup, setup_to_desc
from common import base_fiber, make_tx, rel_l2, scalar_tx as _scalar_tx

GAIN_DB = 16.0
G16 = 10 ** (GAIN_DB / 10)


def _scalar_setup(nsymb, nt, nch, flag, pavg=4.0, length=1e5, dphimax=3e-3):
    gs = _scalar_tx(nsymb, nt, nch, pavg=pavg)
    s = fiber_setup(base_fiber(length=length, dphimax=dphimax, slope=0.057), flag)
    assert not s.isv
    return gs, s


def _scalar_forward(u, s, nspan, gain):
    """noise-free scalar link of the oracle: nspan x [scalar_ssfm ; u*sqrt(gain)] -> (u, steps of every span)"""
    steps = []
    for _ in range(nspan):
        u, st = dso.scalar_ssfm_steps(u, s.betat, s.dzmaxt, s.dphimaxt, s.gam, s.alphalin, s.nfft, s.nfc, s.length, s.fls)
        steps.append(st)
        if gain is not None:
            u = u * math.sqrt(gain)
    return u, steps


def _scalar_oracle(u, s, real=np.float64, **kw):
    return dso.dbp_scalar(u, s.betat, s.gam, s.alphalin, s.nfc, s.length, spm=s.fls[2], xpm=s.fls[3], real=real, **kw)


def _rel(a, b):
    return float(np.linalg.norm(np.asarray(a) - np.asarray(b)) / np.linalg.norm(np.asarray(b)))


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize('nsymb,nt,nch,flag', [(64, 32, 5, 'g-sx'), (64, 32, 5, 'g--x'), (32, 32, 1, 'g-s-')])
def test_scalar_oracle_inverts_the_forward_link(nsymb, nt, nch, flag):
    """forward scalar_ssfm over two spans with a 16 dB gain, then scalar DBP with the forward steps and xi = 1: the Tx
    field back, cross-phase modulation included; the replayed forward run is the pinned scalar_ssfm bit for bit"""
    gs, s = _scalar_setup(nsymb, nt, nch, flag, pavg=8.0)
    fd, nc, ref = orc.scalar_ssfm(gs.FIELDX, s.betat, s.dzmaxt, s.dphimaxt, s.gam, s.alphalin, s.nfft, s.nfc, s.length,
                                  s.fls, 0, None)
    u1, st1 = dso.scalar_ssfm_steps(gs.FIELDX, s.betat, s.dzmaxt, s.dphimaxt, s.gam, s.alphalin, s.nfft, s.nfc, s.length,
                                    s.fls)
    assert np.array_equal(u1, ref) and len(st1) == nc and st1[0] == fd
    u, steps = _scalar_forward(gs.FIELDX, s, 2, G16)
    assert sum(len(x) for x in steps) > 4
    b = _scalar_oracle(u, s, nspan=2, gain=G16, step_len=np.concatenate(steps), span_steps=[len(x) for x in steps])
    err = _rel(b, gs.FIELDX)
    assert err <= 1e-12, err


@pytest.mark.parametrize('flag', ['g-sx', 'g-s-'])
def test_scalar_oracle_converges_with_the_steps(flag):
    """one noise-free nonlinear span: the residual against Tx falls from 1 to 4 to 16 uniform steps and stays below the
    residual of the linear compensation alone (xi = 0)"""
    gs, s = _scalar_setup(64, 32, 5 if flag[3] == 'x' else 1, flag, pavg=4.0)
    u, _ = _scalar_forward(gs.FIELDX, s, 1, None)
    res = [_rel(_scalar_oracle(u, s, steps_per_span=m), gs.FIELDX) for m in (1, 4, 16)]
    lin = _rel(_scalar_oracle(u, s, steps_per_span=1, xi=0.0), gs.FIELDX)
    assert res[0] > res[1] > res[2], res
    assert max(res) < lin, (res, lin)


@pytest.mark.parametrize('nch', [3, 5])
def test_full_field_dbp_beats_spm_only_on_the_centre_channel(nch):
    """a 'g-sx' WDM link: backpropagating the whole multiplex with its XPM ('g-sx') leaves a smaller residual on the
    centre channel than backpropagating each channel's SPM alone ('g-s-'), both with 8 uniform steps per span"""
    gs, s = _scalar_setup(64, 32, nch, 'g-sx', pavg=4.0)
    u, _ = _scalar_forward(gs.FIELDX, s, 2, G16)
    c = nch // 2
    full = _scalar_oracle(u, s, nspan=2, gain=G16, steps_per_span=8)
    s_spm = fiber_setup(base_fiber(length=1e5, dphimax=3e-3, slope=0.057), 'g-s-')
    spm = _scalar_oracle(u, s_spm, nspan=2, gain=G16, steps_per_span=8)
    e_full, e_spm = _rel(full[:, c], gs.FIELDX[:, c]), _rel(spm[:, c], gs.FIELDX[:, c])
    print('centre channel of %d: residual full-field DBP %.3e, SPM-only DBP %.3e' % (nch, e_full, e_spm))
    assert e_full < 0.5 * e_spm, (e_full, e_spm)


def _create_rc(desc, d):
    lib = _lib.load()
    rc = lib.pmx_dbp_create(None, ctypes.byref(desc), ctypes.byref(d), ctypes.byref(ctypes.c_void_p()))
    return rc, lib.pmx_last_error(None).decode()


def test_dbp_create_rejects_what_no_route_runs():
    """without a context: PMX_ERR_UNSUPPORTED with a message naming the limit for the scalar path above 2^12 or with 9
    columns, nfft 2^5, and 9 columns below 2^12; a valid small scalar descriptor gets as far as the missing context"""
    d, dk = _lib.make_dbp(2, G16, steps_per_span=4)
    _scalar_setup(256, 32, 1, 'g-sx')                                     # scalar 2^13
    desc, keep = setup_to_desc(fiber_setup(base_fiber(length=1e5), 'g-sx'))
    rc, msg = _create_rc(desc, d)
    assert rc == _lib.PMX_ERR_UNSUPPORTED and 'scalar path' in msg and '2^12' in msg, msg
    _scalar_setup(32, 32, 9, 'g-sx')                                      # scalar, 9 columns of 2^10
    desc, keep = setup_to_desc(fiber_setup(base_fiber(length=1e5), 'g-sx'))
    rc, msg = _create_rc(desc, d)
    assert rc == _lib.PMX_ERR_UNSUPPORTED and 'nfc=9' in msg and '8 columns' in msg, msg
    _scalar_setup(32, 32, 1, 'g-sx')                                      # valid: 2^10 scalar
    desc, keep = setup_to_desc(fiber_setup(base_fiber(length=1e5), 'g-sx'))
    rc, msg = _create_rc(desc, d)
    assert rc == _lib.PMX_ERR_INVALID and 'null context' in msg, msg
    desc.nfft = 32                                                        # 2^5
    rc, msg = _create_rc(desc, d)
    assert rc == _lib.PMX_ERR_UNSUPPORTED and '2^6' in msg, msg
    make_tx(64, 16, nch=9, ftype='sepfields')                             # two polarizations, 9 columns of 2^10
    desc, keep = setup_to_desc(fiber_setup(base_fiber(), 'g-s-'))
    rc, msg = _create_rc(desc, d)
    assert rc == _lib.PMX_ERR_UNSUPPORTED and 'nfc=9' in msg and '2^12' in msg, msg
    make_tx(64, 16, nch=8, ftype='sepfields')                             # 8 columns are fine
    desc, keep = setup_to_desc(fiber_setup(base_fiber(), 'g-s-'))
    rc, msg = _create_rc(desc, d)
    assert rc == _lib.PMX_ERR_INVALID and 'null context' in msg, msg


def test_dbp_keeps_the_two_polarization_xpm_error():
    make_tx(64, 16, nch=3, ftype='sepfields')
    desc, keep = setup_to_desc(fiber_setup(base_fiber(), 'g-sx'))
    d, dk = _lib.make_dbp(1, 0.0, steps_per_span=2)
    rc, msg = _create_rc(desc, d)
    assert rc == _lib.PMX_ERR_XPM_VECTOR, msg
    with pytest.raises(NotImplementedError):
        pmx.dbp(base_fiber(), 'g-sx')


# ---------------------------------------------------------------------------------------------------------------- GPU
def _cols(a):
    return np.ascontiguousarray(np.asarray(a).T)[None]          # GSTATE [nfft, nfc] -> [1][nfc][nfft]


def _run_device(ctx, s, xs, ys, precision='f64', plates=None, **kw):
    """DBP of the fields xs, ys ([batch][nfc][nfft]) on the device -> (x, y) of the same shape"""
    b = xs.shape[0]
    fld = _lib.DeviceField(ctx, s.nfft, s.nfc, b, precision={'f64': _lib.PMX_F64, 'f32': _lib.PMX_F32}[precision])
    fld.upload(xs, ys)
    plan = dbp_plan(ctx, s, batch=b, precision=precision, plates=plates, **kw)
    launches = ctx.launches
    plan.execute(fld)
    assert ctx.launches == launches + 1                          # the whole link in one launch
    plan.close()
    out = fld.download()
    fld.close()
    return out


def _explicit(s, nspan, seed):
    rng = np.random.default_rng(seed)
    steps = [list(np.diff(np.concatenate([[0.0], np.sort(rng.random(2 + k)) * s.length, [s.length]]))) for k in range(nspan)]
    return dict(step_len=np.concatenate(steps), span_steps=[len(x) for x in steps])


TWO_POL = [  # nch, manakov, schedule, nspan
    (1, False, 'uniform', 3),
    (3, True, 'explicit', 1),
    (8, False, 'explicit', 3),
    (1, True, 'uniform', 1),
]


@pytest.mark.gpu
@pytest.mark.parametrize('case', TWO_POL, ids=lambda c: 'nfc%d-%s-%s-%dspan' % (c[0], 'man' if c[1] else 'cnlse', c[2], c[3]))
@pytest.mark.parametrize('lg', [6, 7, 8, 9, 10, 11])
def test_two_pol_dbp_matches_the_oracle_at_every_small_size(ctx, lg, case):
    nch, manakov, sched, nspan = case
    nt = 8 if lg < 9 else 16
    gs = make_tx((1 << lg) // nt, nt, nch=nch, ftype='sepfields' if nch > 1 else 'unique', pavg_mw=4.0)
    s = fiber_setup(base_fiber(length=8e4, slope=0.057, dphimax=0.02), 'g-s-')
    s.manakov = manakov
    g = G16 if nspan > 1 else None
    kw = dict(steps_per_span=4) if sched == 'uniform' else _explicit(s, nspan, lg + nspan)
    gx, gy = _run_device(ctx, s, _cols(gs.FIELDX), _cols(gs.FIELDY), nspan=nspan, gain_db=GAIN_DB if g else None, **kw)
    wx, wy = dbp_oracle.dbp(gs.FIELDX, gs.FIELDY, s.betat, s.gam, s.alphalin, s.nfc, s.length,
                            'yes' if manakov else 'no', nspan=nspan, gain=g, **kw)
    err = rel_l2(gx[0].T, gy[0].T, wx, wy)
    print('small dbp parity 2^%d %s: rel_l2 %.3e' % (lg, case, err))
    assert err <= 1e-10


def _pmd_setup(nsymb, nt, nplates, manakov, nch=1):
    gs = make_tx(nsymb, nt, nch=nch, ftype='sepfields' if nch > 1 else 'unique', pavg_mw=4.0)
    fib = base_fiber(length=8e4, slope=0.057, dphimax=0.02, dgd=0.5, nplates=nplates, manakov='yes' if manakov else 'no')
    s = fiber_setup(fib, 'gps-', rng=np.random.Generator(np.random.PCG64(7)))
    return gs, s


def _pmd_brfs(s, nspan, batch=1):
    """[span][realization] plate draws: the setup's own plates first, fresh draws for the rest"""
    out = []
    for k in range(nspan):
        row = []
        for b in range(batch):
            if k == 0 and b == 0:
                row.append({x: np.asarray(s.brf[x], dtype=np.float64) for x in ('db0', 'theta', 'epsilon')})
            else:
                row.append(dict(zip(('db0', 'theta', 'epsilon'), mc.draw_plates(mc.plate_seed(b, k), s.nplates))))
        out.append(row)
    return out


def _pmd_plates(brfs):
    return tuple(np.array([[b[x] for b in row] for row in brfs]) for x in ('db0', 'theta', 'epsilon'))


PMD = [  # nsymb, nt, manakov, schedule, nspan, batch, nplates
    (32, 8, True, 'one_step', 1, 1, 20),
    (32, 8, False, 'explicit', 2, 2, 20),
    (64, 16, False, 'one_step', 2, 2, 20),
    (64, 16, True, 'uniform', 3, 1, 12),
]


@pytest.mark.gpu
@pytest.mark.parametrize('case', PMD, ids=lambda c: '%dx%d-%s-%s-%dspan-b%d-%dpl' % (c[0], c[1], 'man' if c[2] else 'cnlse', c[3], c[4], c[5], c[6]))
def test_pmd_dbp_matches_the_oracle_small(ctx, case):
    nsymb, nt, manakov, sched, nspan, batch, nplates = case
    gs, s = _pmd_setup(nsymb, nt, nplates, manakov)
    g = G16 if nspan > 1 else None
    kw = dict(steps_per_span=1) if sched == 'one_step' else (dict(steps_per_span=5) if sched == 'uniform'
                                                              else _explicit(s, nspan, nsymb + nspan))
    brfs = _pmd_brfs(s, nspan, batch)                                   # per-realization plates when batch > 1
    xs = np.concatenate([_cols(gs.FIELDX), _cols(np.roll(gs.FIELDX, 7, axis=0) * 1j)][:batch])
    ys = np.concatenate([_cols(gs.FIELDY), _cols(np.roll(gs.FIELDY, -5, axis=0))][:batch])
    gx, gy = _run_device(ctx, s, xs, ys, plates=_pmd_plates(brfs), nspan=nspan, gain_db=GAIN_DB if g else None, **kw)
    errs = []
    for b in range(batch):
        wx, wy = dpo.dbp_pmd(xs[b].T, ys[b].T, s.betat, s.db1, s.gam, s.alphalin, s.nfc, s.length,
                             'yes' if manakov else 'no', [row[b] for row in brfs], nspan=nspan, gain=g, **kw)
        errs.append(rel_l2(gx[b].T, gy[b].T, wx, wy))
    print('small dbp pmd parity %s: rel_l2 %s' % (case, ['%.3e' % e for e in errs]))
    assert max(errs) <= 1e-10, errs


# Launch powers [mW per channel] keep each case well conditioned: DBP with few long steps of a strongly nonlinear WDM
# link amplifies a rounding difference (measured with the oracle alone: a 1e-15 relative perturbation of the input of
# the 'g--x' case grows to 1.9e-9 at 8 mW and to 2e-12 at 2 mW), which would measure the link, not the kernel.
SCALAR = [  # nsymb, nt, nch, flag, nspan, schedule, launch power
    (32, 32, 1, 'g-sx', 2, 'uniform', 8.0),     # ex06_ber.m
    (64, 32, 5, 'g-sx', 2, 'explicit', 8.0),    # ex10_wdm.m
    (64, 32, 5, 'g--x', 1, 'uniform', 2.0),
    (16, 16, 8, 'g-sx', 2, 'explicit', 4.0),    # 8 columns at 2^8
    (128, 32, 1, 'g-s-', 2, 'uniform', 8.0),    # 2^12
    (128, 32, 2, 'g-sx', 1, 'explicit', 4.0),   # 2^12, transposed resident layout, two columns
]


@pytest.mark.gpu
@pytest.mark.parametrize('case', SCALAR, ids=lambda c: '%dx%dx%d-%s-%dspan-%s-%gmW' % c)
def test_scalar_dbp_matches_the_oracle(ctx, case):
    nsymb, nt, nch, flag, nspan, sched, pavg = case
    gs, s = _scalar_setup(nsymb, nt, nch, flag, pavg=pavg)
    g = G16 if nspan > 1 else None
    kw = dict(steps_per_span=6) if sched == 'uniform' else _explicit(s, nspan, nsymb + nch)
    u = pmx.GSTATE.FIELDX
    gx, _ = _run_device(ctx, s, _cols(u), np.zeros_like(_cols(u)), nspan=nspan, gain_db=GAIN_DB if g else None, **kw)
    w = _scalar_oracle(u, s, nspan=nspan, gain=g, **kw)
    err = _rel(gx[0].T, w)
    print('scalar dbp parity %s: rel_l2 %.3e' % (case, err))
    assert err <= 1e-10


@pytest.mark.gpu
@pytest.mark.parametrize('case', ['2pol_2e10_g-s-', 'ex10_g-sx', '2pol_2e11_gps-'])
def test_dbp_inverts_fiber_on_the_device_small(case):
    """pmx.fiber(fib, flag, trace=True) then pmx.dbp(fib, flag, step_len=trace_dz): the Tx field back"""
    G = pmx.GSTATE
    brf_kw = {}
    if case == '2pol_2e10_g-s-':
        make_tx(64, 16, pavg_mw=8.0)
        fib, flag = base_fiber(length=1e5, dphimax=0.01), 'g-s-'
    elif case == 'ex10_g-sx':
        _scalar_tx(64, 32, 5, pavg=8.0)
        fib, flag = base_fiber(length=1e5, dphimax=3e-3, slope=0.057), 'g-sx'
    else:
        make_tx(128, 16, pavg_mw=8.0)
        fib, flag = base_fiber(length=8e4, dphimax=0.01, dgd=0.5, nplates=20, manakov='yes'), 'gps-'
    tx = G.FIELDX.copy()
    ty = G.FIELDY.copy() if G.has_y() else None
    brf = pmx.fiber(fib, flag, rng=np.random.Generator(np.random.PCG64(3)), trace=True)
    dz = pmx.FIBER_LAST['trace_dz']
    assert len(dz) == pmx.FIBER_LAST['ncycle'] > 1
    if flag[1] == 'p':
        brf_kw = dict(brf=brf)
    pmx.dbp(fib, flag, step_len=dz, **brf_kw)
    err = rel_l2(G.FIELDX, G.FIELDY, tx, ty) if ty is not None else _rel(G.FIELDX, tx)
    print('small dbp exact inverse %s: %d steps, rel_l2 %.3e' % (case, len(dz), err))
    assert err <= 1e-11


@pytest.mark.gpu
@pytest.mark.parametrize('what', ['two_pol', 'scalar'])
def test_small_dbp_fp32(ctx, what):
    if what == 'two_pol':
        gs = make_tx(64, 16, pavg_mw=4.0)
        s = fiber_setup(base_fiber(length=8e4, slope=0.057, dphimax=0.02), 'g-s-')
        gx, gy = _run_device(ctx, s, _cols(gs.FIELDX), _cols(gs.FIELDY), precision='f32', nspan=2, gain_db=GAIN_DB,
                             steps_per_span=20)
        wx, wy = dbp_oracle.dbp(gs.FIELDX, gs.FIELDY, s.betat, s.gam, s.alphalin, s.nfc, s.length, 'no', nspan=2, gain=G16,
                                steps_per_span=20)
        err = rel_l2(gx[0].T, gy[0].T, wx, wy)
    else:
        gs, s = _scalar_setup(32, 32, 1, 'g-sx', pavg=1.0)        # ex06 shape, well conditioned (see SCALAR)
        u = pmx.GSTATE.FIELDX
        gx, _ = _run_device(ctx, s, _cols(u), np.zeros_like(_cols(u)), precision='f32', nspan=2, gain_db=GAIN_DB,
                            steps_per_span=20)
        err = _rel(gx[0].T, _scalar_oracle(u, s, nspan=2, gain=G16, steps_per_span=20))
    print('small dbp fp32 %s: rel_l2 %.3e' % (what, err))
    assert err <= 1e-5


@pytest.mark.gpu
def test_small_dbp_realizations_are_independent(ctx):
    """a batch of 5 realizations with per-realization plates equals, bit for bit, each realization run alone"""
    gs, s = _pmd_setup(64, 16, 20, True, nch=1)
    brfs = _pmd_brfs(s, 2, 5)
    xs = np.concatenate([_cols(np.roll(gs.FIELDX, 11 * b, axis=0)) for b in range(5)])
    ys = np.concatenate([_cols(np.roll(gs.FIELDY, -3 * b, axis=0)) for b in range(5)])
    kw = dict(nspan=2, gain_db=GAIN_DB, steps_per_span=3)
    bx, by = _run_device(ctx, s, xs, ys, plates=_pmd_plates(brfs), **kw)
    for b in range(5):
        one = [[row[b]] for row in brfs]
        ox, oy = _run_device(ctx, s, xs[b:b + 1], ys[b:b + 1], plates=_pmd_plates(one), **kw)
        assert np.array_equal(ox[0], bx[b]) and np.array_equal(oy[0], by[b]), b
