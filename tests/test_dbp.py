"""Digital backpropagation (pmx_dbp_create / pmx_dbp_exec, polmux_b200.dbp, tests/dbp_oracle.py).

The reference has no DBP: the oracle is the numpy restatement in tests/dbp_oracle.py, tied to the pinned forward
oracle by one property -- run with the forward run's own steps, xi = 1 and no noise or PMD, DBP returns the transmitted
field up to rounding."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

import oracle.fiber_oracle as orc
import dbp_oracle
import polmux_b200 as pmx
from polmux_b200 import _lib, mc, synth
from polmux_b200.dbp import dbp_plan
from polmux_b200.fiber import fiber_setup, setup_to_desc
from common import base_fiber, make_tx, rel_l2

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GAIN_DB = 16.0


def _setup(nsymb, nt, nch=1, ftype='unique', pavg_mw=4.0, length=8e4, manakov=False, slope=0.057):
    """-> (oracle GState with the Tx field, product FiberSetup of the 'g-s-' fiber; GSTATE holds the same Tx field)"""
    gs = make_tx(nsymb, nt, nch=nch, ftype=ftype, pavg_mw=pavg_mw)
    fib = base_fiber(length=length, slope=slope, dphimax=0.02)
    s = fiber_setup(fib, 'g-s-')
    s.manakov = manakov
    return gs, s


def _forward(gs, s, nspan, gain):
    """noise-free link of the oracle: nspan x [matrix_ssfm ; u*sqrt(gain)] -> (ux, uy, steps of every span)"""
    ux, uy, steps = gs.FIELDX.copy(), gs.FIELDY.copy(), []
    for _ in range(nspan):
        _, _, ux, uy, _, sched = orc.matrix_ssfm(ux, uy, s.betat, s.db1, s.dzmaxt, s.dphimaxt, s.gam, s.alphalin, s.nfc,
                                                 s.length, 1, 'yes' if s.manakov else 'no', s.fls, s.brf)
        steps.append([st['dz'] for st in sched])
        if gain is not None:
            ux, uy = ux * math.sqrt(gain), uy * math.sqrt(gain)
    return ux, uy, steps


def _oracle_dbp(ux, uy, s, real=np.float64, **kw):
    return dbp_oracle.dbp(ux, uy, s.betat, s.gam, s.alphalin, s.nfc, s.length, 'yes' if s.manakov else 'no', real=real, **kw)


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize('manakov', [False, True])
@pytest.mark.parametrize('nch', [1, 3])
def test_oracle_dbp_inverts_the_forward_link(manakov, nch):
    """forward 'g-s-' over two spans with a 16 dB gain, then DBP with the forward schedule and xi = 1: the Tx field back"""
    gs, s = _setup(256, 16, nch=nch, ftype='sepfields' if nch > 1 else 'unique', manakov=manakov)
    assert s.scalars['b30'] != 0.0
    g = 10 ** (GAIN_DB / 10)
    ux, uy, steps = _forward(gs, s, 2, g)
    assert sum(len(x) for x in steps) > 4
    bx, by = _oracle_dbp(ux, uy, s, nspan=2, gain=g, step_len=np.concatenate(steps), span_steps=[len(x) for x in steps])
    assert rel_l2(bx, by, gs.FIELDX, gs.FIELDY) <= 1e-12


@pytest.mark.parametrize('manakov', [False, True])
def test_oracle_dbp_converges_with_the_steps(manakov):
    """one noise-free nonlinear span: the residual against Tx falls from 1 to 4 to 16 uniform steps and stays below the
    residual of the linear compensation alone (xi = 0)"""
    gs, s = _setup(256, 16, pavg_mw=30.0, manakov=manakov)
    ux, uy, _ = _forward(gs, s, 1, None)
    res = [rel_l2(*_oracle_dbp(ux, uy, s, steps_per_span=m), gs.FIELDX, gs.FIELDY) for m in (1, 4, 16)]
    lin = rel_l2(*_oracle_dbp(ux, uy, s, steps_per_span=1, xi=0.0), gs.FIELDX, gs.FIELDY)
    assert res[0] > res[1] > res[2], res
    assert max(res) < lin, (res, lin)


def test_dbp_structs_match_the_header(tmp_path):
    """gcc probe against the header: pmx_dbp_desc and the extended pmx_mc_receiver equal their ctypes mirrors"""
    structs = {'pmx_dbp_desc': _lib.DbpDesc, 'pmx_mc_receiver': _lib.McReceiver}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "polmux_ssfm.h"', 'int main(void){']
    for cname, cls in structs.items():
        lines.append('printf("%s %%zu\\n", sizeof(%s));' % (cname, cname))
        for fname, _ in cls._fields_:
            lines.append('printf("%s.%s %%zu\\n", offsetof(%s, %s));' % (cname, fname, cname, fname))
    lines.append('return 0;}')
    src = tmp_path / 'probe.c'
    src.write_text('\n'.join(lines))
    exe = tmp_path / 'probe'
    subprocess.run(['gcc', '-I', os.path.join(ROOT, 'include'), str(src), '-o', str(exe)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    for cname, cls in structs.items():
        assert int(out[cname]) == ctypes.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert int(out['%s.%s' % (cname, fname)]) == getattr(cls, fname).offset, (cname, fname)
    assert _lib.McReceiver.dbp.offset == ctypes.sizeof(_lib.McReceiver) - ctypes.sizeof(ctypes.c_void_p)   # appended


@pytest.mark.skipif(_lib.load().pmx_device_count() > 0, reason='a GPU is present')
def test_dbp_has_no_cpu_fallback():
    make_tx(256, 16)
    with pytest.raises(_lib.PolmuxError):
        pmx.dbp(base_fiber(), 'g-s-', steps_per_span=2)


def test_dbp_create_rejects_invalid_schedules():
    """pmx_dbp_create checks its descriptors before it needs a context: PMX_ERR_INVALID with a message for each"""
    lib = _lib.load()
    make_tx(256, 16)
    s = fiber_setup(base_fiber(), 'g-s-')
    desc, keep = setup_to_desc(s)
    L = s.length
    bad = {
        'negative': dict(step_len=[L / 2 + 1.0, -1.0, L / 2]),
        'not finite': dict(step_len=[L / 2, float('nan'), L / 2]),
        'sum to': dict(step_len=[L / 2, L / 4]),
        'nspan': dict(nspan=0, steps_per_span=2),
        'xi': dict(steps_per_span=2, xi=float('inf')),
        'gain': dict(steps_per_span=2, gain=-1.0),
    }
    for what, kw in bad.items():
        kw = dict(kw)
        d, dk = _lib.make_dbp(kw.pop('nspan', 1), kw.pop('gain', 0.0), **kw)
        h = ctypes.c_void_p()
        rc = lib.pmx_dbp_create(None, ctypes.byref(desc), ctypes.byref(d), ctypes.byref(h))
        assert rc == _lib.PMX_ERR_INVALID, what
        assert what in lib.pmx_last_error(None).decode(), (what, lib.pmx_last_error(None))
    d, dk = _lib.make_dbp(2, 40.0, step_len=[L / 4] * 4)     # valid: only the missing context is left to complain about
    assert lib.pmx_dbp_create(None, ctypes.byref(desc), ctypes.byref(d), ctypes.byref(ctypes.c_void_p())) == _lib.PMX_ERR_INVALID
    assert 'null context' in lib.pmx_last_error(None).decode()


def test_genie_receiver_takes_no_dbp():
    make_tx(256, 16)
    s = fiber_setup(base_fiber(), 'g-s-')
    with pytest.raises(ValueError):
        mc.McRunner(None, s, None, None, np.zeros((2, 256), np.uint8), 256, 16, 1, 16.0, 5.0, 2, 2, receiver='genie',
                    compensation='dbp')


# ---------------------------------------------------------------------------------------------------------------- GPU
def _run_device(ctx, s, xs, ys, precision='f64', **kw):
    """DBP of the fields xs, ys ([batch][nfc][nfft]) on the device -> (x, y) of the same shape"""
    b = xs.shape[0]
    fld = _lib.DeviceField(ctx, s.nfft, s.nfc, b, precision={'f64': _lib.PMX_F64, 'f32': _lib.PMX_F32}[precision])
    fld.upload(xs, ys)
    plan = dbp_plan(ctx, s, batch=b, precision=precision, **kw)
    plan.execute(fld)
    plan.close()
    out = fld.download()
    fld.close()
    return out


def _cols(a):
    return np.ascontiguousarray(np.asarray(a).T)[None]          # GSTATE [nfft, nfc] -> [1][nfc][nfft]


PARITY = [  # nsymb, nt, nch, manakov, schedule, nspan, batch
    (256, 16, 1, False, 'uniform', 3, 1),
    (256, 16, 3, True, 'explicit', 1, 1),
    (4096, 16, 1, True, 'explicit', 3, 1),
    (4096, 16, 3, False, 'uniform', 1, 1),
    (65536, 16, 1, True, 'uniform', 1, 2),
    (65536, 16, 1, False, 'explicit', 3, 2),
]


@pytest.mark.gpu
@pytest.mark.parametrize('case', PARITY, ids=lambda c: '%dx%d-nfc%d-%s-%s-%dspan-b%d' % (c[0], c[1], c[2], 'man' if c[3] else 'cnlse', c[4], c[5], c[6]))
def test_dbp_matches_the_oracle_fp64(ctx, case):
    nsymb, nt, nch, manakov, sched, nspan, batch = case
    gs, s = _setup(nsymb, nt, nch=nch, ftype='sepfields' if nch > 1 else 'unique', manakov=manakov)
    g = 10 ** (GAIN_DB / 10) if nspan > 1 else None
    if sched == 'uniform':
        kw = dict(steps_per_span=4)
    else:
        rng = np.random.default_rng(nsymb + nspan)
        steps = [list(np.diff(np.concatenate([[0.0], np.sort(rng.random(2 + k)) * s.length, [s.length]]))) for k in range(nspan)]
        kw = dict(step_len=np.concatenate(steps), span_steps=[len(x) for x in steps])
    xs = np.concatenate([_cols(gs.FIELDX), _cols(np.roll(gs.FIELDX, 7, axis=0) * 1j)][:batch])
    ys = np.concatenate([_cols(gs.FIELDY), _cols(np.roll(gs.FIELDY, -5, axis=0))][:batch])
    gx, gy = _run_device(ctx, s, xs, ys, nspan=nspan, gain_db=GAIN_DB if g else None, **kw)
    errs = []
    for b in range(batch):
        wx, wy = _oracle_dbp(xs[b].T, ys[b].T, s, nspan=nspan, gain=g, **kw)
        errs.append(rel_l2(gx[b].T, gy[b].T, wx, wy))
    print('dbp parity %s: rel_l2 %s' % (case, ['%.3e' % e for e in errs]))
    assert max(errs) <= 1e-10, errs


@pytest.mark.gpu
@pytest.mark.parametrize('manakov', [False, True])
def test_dbp_matches_the_oracle_fp32(ctx, manakov):
    gs, s = _setup(4096, 16, manakov=manakov)
    g = 10 ** (GAIN_DB / 10)
    gx, gy = _run_device(ctx, s, _cols(gs.FIELDX), _cols(gs.FIELDY), precision='f32', nspan=2, gain_db=GAIN_DB,
                         steps_per_span=20)
    wx, wy = _oracle_dbp(gs.FIELDX, gs.FIELDY, s, nspan=2, gain=g, steps_per_span=20)
    err = rel_l2(gx[0].T, gy[0].T, wx, wy)
    print('dbp parity fp32 manakov=%s: rel_l2 %.3e' % (manakov, err))
    assert err <= 1e-5


@pytest.mark.gpu
def test_dbp_inverts_fiber_on_the_device_c1():
    """pmx.fiber(fib, 'g-s-', trace=True) then pmx.dbp(fib, 'g-s-', step_len=trace_dz): the Tx field back (C1 size,
    2^16, CNLSE, 100 km)"""
    make_tx(4096, 16)
    G = pmx.GSTATE
    tx, ty = G.FIELDX_TX.copy(), G.FIELDY_TX.copy()
    fib = base_fiber(length=1e5)
    pmx.fiber(fib, 'g-s-', trace=True)
    assert pmx.FIBER_LAST['ncycle'] > 1
    pmx.dbp(fib, 'g-s-', step_len=pmx.FIBER_LAST['trace_dz'])
    err = rel_l2(G.FIELDX, G.FIELDY, tx, ty)
    print('dbp exact inverse C1: %d steps, rel_l2 %.3e' % (pmx.FIBER_LAST['ncycle'], err))
    assert err <= 1e-11


@pytest.mark.gpu
def test_dbp_inverts_a_manakov_span_on_the_device_c2(ctx):
    """the same on a C2 span: 2^20, Manakov, 80 km, through the resident plan API"""
    from polmux_b200.fiber import setup_to_desc
    make_tx(65536, 16)
    G = pmx.GSTATE
    s = fiber_setup(base_fiber(length=8e4), 'g-s-')
    s.manakov = True
    desc, keep = setup_to_desc(s)
    fld = _lib.DeviceField(ctx, s.nfft, 1, 1)
    fld.upload(G.FIELDX_TX, G.FIELDY_TX)
    plan = _lib.Plan(ctx, desc, keep)
    res = plan.execute(fld, trace_cap=1 << 16)
    plan.close()
    dz, _ = res.schedule(0)
    dbp_plan(ctx, s, step_len=dz).execute(fld)
    x, y = fld.download()
    fld.close()
    err = rel_l2(x[0, 0], y[0, 0], G.FIELDX_TX[:, 0], G.FIELDY_TX[:, 0])
    print('dbp exact inverse C2 span: %d steps, rel_l2 %.3e' % (len(dz), err))
    assert len(dz) > 1 and err <= 1e-11


@pytest.mark.gpu
def test_dbp_realizations_are_independent(ctx):
    """DBP of a batch equals, bit for bit, DBP of each realization alone (2^20: the batch runs as two stream groups)"""
    gs, s = _setup(65536, 16, manakov=True)
    xs = np.concatenate([_cols(np.roll(gs.FIELDX, 11 * b, axis=0)) for b in range(3)])
    ys = np.concatenate([_cols(np.roll(gs.FIELDY, -3 * b, axis=0)) for b in range(3)])
    kw = dict(nspan=2, gain_db=GAIN_DB, steps_per_span=2)
    bx, by = _run_device(ctx, s, xs, ys, **kw)
    for b in range(3):
        ox, oy = _run_device(ctx, s, xs[b:b + 1], ys[b:b + 1], **kw)
        assert np.array_equal(ox[0], bx[b]) and np.array_equal(oy[0], by[b]), b


def _mc_scenario(nsymb, nt, pavg_mw):
    ex, ey, sx, sy = synth.pdm_qpsk(nsymb, nt, 1)
    pmx.reset_all(nsymb, nt, 1)
    G = pmx.GSTATE
    G.SYMBOLRATE, G.LAMBDA, G.POWER = 28.0, np.array([1550.0]), np.array([float(pavg_mw)])
    pmx.create_field('unique', ex, ey, {'power': 'average'})
    fib = dict(synth.SMF)
    fib.update(length=8e4, dgd=0.3, nplates=20, manakov='yes')
    setup = fiber_setup(fib, 'gps-', rng=np.random.Generator(np.random.PCG64(0)))
    return G, setup, np.stack([sx[:, 0], sy[:, 0]]).astype(np.uint8)


@pytest.mark.gpu
def test_mc_with_dbp_python_and_native_agree(ctx):
    """McRunner(compensation='dbp') and run_mc_native(..., dbp_params=...) count the same errors, realization by
    realization, on a small seeded job (16 realizations, 2 spans at 2^16); the blind receiver runs behind DBP too"""
    nsymb, nt, nspan, nreal, batch = 1 << 12, 16, 2, 16, 4
    G, setup, sym = _mc_scenario(nsymb, nt, 8.0)
    x = {'oftype': 'gauss', 'obw': 1.9, 'eftype': 'bessel5', 'ebw': 0.65, 'lopower': 0.0}
    dspp = dict(mu=1 / 2000, freqavg=200)
    dbpp = dict(steps_per_span=4)
    r = mc.McRunner(ctx, setup, G.FIELDX_TX, G.FIELDY_TX, sym, nsymb, nt, nspan, 16.0, 5.0, nreal, batch, receiver='cohmix',
                    dsp_params=dspp, rx_params=x, compensation='dbp', dbp_params=dbpp)
    want, _ = r.run(ase_seed=3)
    r.close()
    got, _ = mc.run_mc_native(setup, G.FIELDX_TX, G.FIELDY_TX, sym, nsymb, nt, nspan, 16.0, 5.0, nreal, batch, devices=(0,),
                              ase_seed=3, receiver=x, dsp_params=dspp, dbp_params=dbpp)
    print('mc dbp counts', want.tolist())
    assert np.array_equal(got, want), (got, want)
    r = mc.McRunner(ctx, setup, G.FIELDX_TX, G.FIELDY_TX, sym, nsymb, nt, nspan, 16.0, 5.0, nreal, batch, receiver='blind',
                    dsp_params=dspp, compensation='dbp', dbp_params=dbpp)
    blind, _ = r.run(ase_seed=3)
    r.close()
    assert blind.shape == (nreal,) and blind.min() >= 0
