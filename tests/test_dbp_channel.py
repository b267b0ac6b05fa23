"""Single-channel digital backpropagation (pmx_dbp_channel_create, polmux_b200.dbp with ich / decim, McRunner with
dbp_params 'decim'): one channel of a 'unique' multiplex cut out, backpropagated at nfft/decim samples on its own
dispersion, and returned to its own bins.

Oracle: tests/dbp_oracle.dbp_channel -- the full-field oracles on the cropped spectrum -- tied here to the full-field
oracle (xi = 0: the full DBP followed by the ideal band-pass) and to the forward oracle (the exact inverse of a link run
on the channel alone)."""
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
from polmux_b200.receiver import CohmixSetup, channel_ndfn
from common import _cols, _rel, base_fiber, make_tx, rel_l2

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GAIN_DB = 16.0
G16 = 10 ** (GAIN_DB / 10)


def _setup(nsymb, nt, nch=3, flag='g-s-', manakov=False, pavg_mw=4.0, length=8e4, **extra):
    """-> (oracle GState, FiberSetup): a 'unique' multiplex of nch 28-GBaud channels at 50 GHz in GSTATE"""
    gs = make_tx(nsymb, nt, nch=nch, ftype='unique', pavg_mw=pavg_mw)
    fib = base_fiber(length=length, slope=0.057, dphimax=0.02, manakov='yes' if manakov else 'no', **extra)
    s = fiber_setup(fib, flag, rng=np.random.Generator(np.random.PCG64(7)))
    s.manakov = manakov
    return gs, s


def _oracle(ux, uy, s, shift, decim, **kw):
    return dbp_oracle.dbp_channel(ux, uy, s.betat, s.gam, s.alphalin, s.length, 'yes' if s.manakov else 'no', shift, decim,
                                  **kw)


def _scalar_unique(nsymb, nt, nch, pavg=4.0):
    """GSTATE <- a single-polarization 'unique' multiplex (FIELDY empty) of nch channels"""
    ex, _, _, _ = synth.pdm_qpsk(nsymb, nt, nch)
    pmx.reset_all(nsymb, nt, nch)
    G = pmx.GSTATE
    G.SYMBOLRATE, G.LAMBDA, G.POWER = 28.0, synth.wdm_lambdas(nch, 1550.0, 0.4), np.full(nch, pavg)
    pmx.create_field('unique', ex, None, {'power': 'average'})
    return G


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_channel_offset_is_the_receivers():
    """channel_ndfn is the ndfn CohmixSetup gives every channel of a 'unique' multiplex, and 0 bins for the centre one"""
    make_tx(256, 16, nch=3)
    x = {'oftype': 'gauss', 'obw': 1.9, 'eftype': 'bessel5', 'ebw': 0.65}
    got = [channel_ndfn(i) for i in (1, 2, 3)]
    assert got == [CohmixSetup(i, x).ndfn for i in (1, 2, 3)]
    assert got[1] == 0 and got[0] == -got[2] != 0


@pytest.mark.parametrize('manakov', [False, True])
def test_oracle_linear_is_the_band_passed_full_field_dbp(manakov):
    """xi = 0: single-channel DBP of an off-centre channel equals full-field DBP followed by the ideal band-pass"""
    gs, s = _setup(256, 16, manakov=manakov)
    m = channel_ndfn(1)
    kw = dict(nspan=2, gain=G16, steps_per_span=3, xi=0.0)
    cx, cy = _oracle(gs.FIELDX, gs.FIELDY, s, m, 8, **kw)
    fx, fy = dbp_oracle.dbp(gs.FIELDX, gs.FIELDY, s.betat, s.gam, s.alphalin, 1, s.length, 'yes' if manakov else 'no', **kw)
    b = dbp_oracle.channel_bins(s.nfft, m, 8)
    err = rel_l2(cx, cy, dbp_oracle.band_pass(fx, b), dbp_oracle.band_pass(fy, b))
    assert err <= 1e-13, err


@pytest.mark.parametrize('flag', ['g-s-', 'gps-'])
def test_oracle_inverts_a_link_run_on_the_channel_alone(flag):
    """forward oracle on the channel alone at M samples (two spans, 16 dB, 'gps-' with other plates in every span),
    embedded at shift 0 in N; single-channel DBP with the forward steps and xi = 1 returns the embedded Tx"""
    gs, s = _setup(256, 16, nch=1, flag=flag, dgd=0.5, nplates=20) if flag == 'gps-' else _setup(256, 16, nch=1)
    r, N = 4, s.nfft
    b = dbp_oracle.channel_bins(N, 0, r)
    tx, ty = dbp_oracle.crop(gs.FIELDX, b, r), dbp_oracle.crop(gs.FIELDY, b, r)
    bt, d1 = s.betat[b], s.db1[b]
    brfs = [dict(s.brf)] * 2                     # (without 'p' the forward oracle still reads the identity plates)
    if flag == 'gps-':
        brfs[1] = dict(zip(('db0', 'theta', 'epsilon'), mc.draw_plates(mc.plate_seed(0, 1), s.nplates)))
    ux, uy, steps = tx, ty, []
    for k in range(2):
        _, _, ux, uy, _, sched = orc.matrix_ssfm(ux, uy, bt, d1, s.dzmaxt, s.dphimaxt, s.gam, s.alphalin, 1, s.length,
                                                 s.nplates, 'no', s.fls, brfs[k])
        steps.append([st['dz'] for st in sched])
        ux, uy = ux * math.sqrt(G16), uy * math.sqrt(G16)
    assert sum(len(x) for x in steps) > 4
    ex, ey = dbp_oracle.embed(ux, b, N, r), dbp_oracle.embed(uy, b, N, r)
    kw = dict(nspan=2, gain=G16, step_len=np.concatenate(steps), span_steps=[len(x) for x in steps])
    if flag == 'gps-':
        kw.update(db1=s.db1, brfs=brfs)
    gx, gy = _oracle(ex, ey, s, 0, r, **kw)
    err = rel_l2(gx, gy, dbp_oracle.embed(tx, b, N, r), dbp_oracle.embed(ty, b, N, r))
    assert err <= 1e-12, err


def test_dbp_band_matches_the_header(tmp_path):
    """gcc probe against the header: pmx_dbp_band equals its ctypes mirror"""
    cls = _lib.DbpBand
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "polmux_ssfm.h"', 'int main(void){',
             'printf("size %zu\\n", sizeof(pmx_dbp_band));']
    lines += ['printf("%s %%zu\\n", offsetof(pmx_dbp_band, %s));' % (f, f) for f, _ in cls._fields_]
    lines.append('return 0;}')
    src = tmp_path / 'probe.c'
    src.write_text('\n'.join(lines))
    exe = tmp_path / 'probe'
    subprocess.run(['gcc', '-I', os.path.join(ROOT, 'include'), str(src), '-o', str(exe)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(out['size']) == ctypes.sizeof(cls)
    for f, _ in cls._fields_:
        assert int(out[f]) == getattr(cls, f).offset, f


def _create_rc(desc, d, shift, decim):
    lib = _lib.load()
    band = _lib.make_band(shift, decim)
    rc = lib.pmx_dbp_channel_create(None, ctypes.byref(desc), ctypes.byref(d), ctypes.byref(band),
                                    ctypes.byref(ctypes.c_void_p()))
    return rc, lib.pmx_last_error(None).decode()


def test_channel_create_validates_before_it_needs_a_context():
    """every refusal comes without a context, with its message; a valid request gets as far as the missing context"""
    d, dk = _lib.make_dbp(2, G16, steps_per_span=4)
    _setup(256, 16)                                                             # 'unique', 2^12, two polarizations
    desc, keep = setup_to_desc(fiber_setup(base_fiber(), 'g-s-'))
    m = channel_ndfn(1)
    for decim, code, what in ((3, _lib.PMX_ERR_INVALID, 'power of two'), (1, _lib.PMX_ERR_INVALID, 'power of two'),
                              (0, _lib.PMX_ERR_INVALID, 'power of two'), (128, _lib.PMX_ERR_INVALID, 'at least 2^6')):
        rc, msg = _create_rc(desc, d, m, decim)
        assert rc == code and what in msg, (decim, rc, msg)
    bad, bk = _lib.make_dbp(0, G16, steps_per_span=4)                            # what pmx_dbp_create rejects
    rc, msg = _create_rc(desc, bad, m, 8)
    assert rc == _lib.PMX_ERR_INVALID and 'nspan' in msg, msg
    rc, msg = _create_rc(desc, d, m, 8)
    assert rc == _lib.PMX_ERR_INVALID and 'null context' in msg, msg
    vdesc, vkeep = setup_to_desc(fiber_setup(base_fiber(), 'g-s-'), disp_mode='vector')
    rc, msg = _create_rc(vdesc, d, m, 8)
    assert rc == _lib.PMX_ERR_INVALID and 'null context' in msg, msg
    make_tx(256, 16, nch=3, ftype='sepfields')                                  # three columns
    desc, keep = setup_to_desc(fiber_setup(base_fiber(), 'g-s-'))
    rc, msg = _create_rc(desc, d, 0, 8)
    assert rc == _lib.PMX_ERR_UNSUPPORTED and 'nfc=3' in msg, msg
    _scalar_unique(1024, 16, 3)                                                 # scalar path, 2^14
    desc, keep = setup_to_desc(fiber_setup(base_fiber(), 'g-s-'))
    assert desc.scalar_field == 1
    rc, msg = _create_rc(desc, d, channel_ndfn(1), 2)                           # M = 2^13
    assert rc == _lib.PMX_ERR_UNSUPPORTED and 'scalar path' in msg and '2^12' in msg, msg
    rc, msg = _create_rc(desc, d, channel_ndfn(1), 4)                           # M = 2^12: fine
    assert rc == _lib.PMX_ERR_INVALID and 'null context' in msg, msg


def test_python_arguments_are_checked():
    make_tx(256, 16, nch=3)
    with pytest.raises(ValueError):
        pmx.dbp(base_fiber(), 'g-s-', ich=1)                                    # ich without decim
    with pytest.raises(ValueError):
        pmx.dbp(base_fiber(), 'g-s-', decim=8)                                  # decim without ich
    with pytest.raises(ValueError):
        pmx.dbp(base_fiber(), 'g-s-', ich=4, decim=8)                           # no such channel
    make_tx(256, 16)
    s = fiber_setup(base_fiber(), 'g-s-')
    with pytest.raises(ValueError):
        mc.McRunner(None, s, None, None, np.zeros((2, 256), np.uint8), 256, 16, 1, 16.0, 5.0, 2, 2, receiver='genie',
                    compensation='dbp_pmd', dbp_params=dict(decim=8))


@pytest.mark.skipif(_lib.load().pmx_device_count() > 0, reason='a GPU is present')
def test_channel_dbp_has_no_cpu_fallback():
    make_tx(256, 16, nch=3)
    with pytest.raises(_lib.PolmuxError):
        pmx.dbp(base_fiber(), 'g-s-', steps_per_span=2, ich=1, decim=8)


# ---------------------------------------------------------------------------------------------------------------- GPU
def _run_device(ctx, s, xs, ys, precision='f64', plates=None, **kw):
    """DBP of the fields xs, ys ([batch][1][nfft]) on the device -> (x, y) of the same shape"""
    b = xs.shape[0]
    fld = _lib.DeviceField(ctx, s.nfft, 1, b, precision={'f64': _lib.PMX_F64, 'f32': _lib.PMX_F32}[precision])
    fld.upload(xs, ys)
    plan = dbp_plan(ctx, s, batch=b, precision=precision, plates=plates, **kw)
    plan.execute(fld)
    plan.close()
    out = fld.download()
    fld.close()
    return out


def _batch2(gs):
    xs = np.concatenate([_cols(gs.FIELDX), _cols(np.roll(gs.FIELDX, 7, axis=0) * 1j)])
    ys = np.concatenate([_cols(gs.FIELDY), _cols(np.roll(gs.FIELDY, -5, axis=0))])
    return xs, ys


PARITY = [  # nsymb, nt, decim, manakov, ich: every pair of routes at N and at M = N/decim
    (64, 16, 4, False, 1),        # 2^10 on-chip  -> 2^8 on-chip
    (512, 32, 16, True, 3),       # 2^14 passes   -> 2^10 on-chip
    (2048, 32, 16, False, 1),     # 2^16 passes   -> 2^12 passes
    (65536, 16, 8, True, 3),      # 2^20 passes   -> 2^17 passes
]


@pytest.mark.gpu
@pytest.mark.parametrize('precision', ['f64', 'f32'])
@pytest.mark.parametrize('case', PARITY, ids=lambda c: '2^%d-r%d-%s-ch%d' % (int(math.log2(c[0] * c[1])), c[2],
                                                                             'man' if c[3] else 'cnlse', c[4]))
def test_channel_dbp_matches_the_oracle(ctx, case, precision):
    nsymb, nt, r, manakov, ich = case
    gs, s = _setup(nsymb, nt, manakov=manakov)
    m = channel_ndfn(ich)
    assert m != 0
    kw = dict(nspan=2, steps_per_span=3)
    xs, ys = _batch2(gs)
    gx, gy = _run_device(ctx, s, xs, ys, precision, gain_db=GAIN_DB, shift=m, decim=r, **kw)
    errs = []
    for b in range(2):
        wx, wy = _oracle(xs[b].T, ys[b].T, s, m, r, gain=G16, **kw)
        errs.append(rel_l2(gx[b].T, gy[b].T, wx, wy))
    print('channel dbp parity %s %s: rel_l2 %s' % (case, precision, ['%.3e' % e for e in errs]))
    assert max(errs) <= (1e-10 if precision == 'f64' else 1e-5), errs


@pytest.mark.gpu
def test_channel_dbp_pmd_matches_the_oracle(ctx):
    """PMD-aware, a plate draw per realization and span (2^14 -> 2^10)"""
    gs, s = _setup(512, 32, flag='gps-', dgd=0.5, nplates=20)
    m, r = channel_ndfn(1), 16
    brfs = [[dict(zip(('db0', 'theta', 'epsilon'), mc.draw_plates(mc.plate_seed(b, k), s.nplates))) for b in range(2)]
            for k in range(2)]
    plates = tuple(np.array([[p[x] for p in row] for row in brfs]) for x in ('db0', 'theta', 'epsilon'))
    kw = dict(nspan=2, steps_per_span=3)
    xs, ys = _batch2(gs)
    gx, gy = _run_device(ctx, s, xs, ys, gain_db=GAIN_DB, shift=m, decim=r, plates=plates, **kw)
    errs = []
    for b in range(2):
        wx, wy = _oracle(xs[b].T, ys[b].T, s, m, r, gain=G16, db1=s.db1, brfs=[brfs[k][b] for k in range(2)], **kw)
        errs.append(rel_l2(gx[b].T, gy[b].T, wx, wy))
    print('channel dbp pmd parity: rel_l2 %s' % ['%.3e' % e for e in errs])
    assert max(errs) <= 1e-10, errs


@pytest.mark.gpu
@pytest.mark.parametrize('flag', ['g-s-', 'gps-'])
def test_channel_dbp_inverts_fiber_on_the_device(flag):
    """pmx.fiber(..., trace=True) on the channel alone at M = 2^12, embedded at N = 2^16; pmx.dbp(..., ich=1, decim=16,
    step_len=trace_dz) -- with brf for 'gps-' -- returns the embedded Tx"""
    nsymb, nt, r = 2048, 2, 16
    make_tx(nsymb, nt)
    G = pmx.GSTATE
    rate, lam, power = G.SYMBOLRATE, G.LAMBDA.copy(), G.POWER.copy()
    tx, ty = G.FIELDX_TX.copy(), G.FIELDY_TX.copy()
    fib = base_fiber(length=1e5, dgd=0.5, nplates=20)
    brf = pmx.fiber(fib, flag, trace=True, rng=np.random.Generator(np.random.PCG64(3)))
    steps = pmx.FIBER_LAST['trace_dz']
    assert len(steps) > 1
    rx, ry = G.FIELDX.copy(), G.FIELDY.copy()
    pmx.reset_all(nsymb, nt * r, 1)
    G.SYMBOLRATE, G.LAMBDA, G.POWER = rate, lam, power
    b = dbp_oracle.channel_bins(nsymb * nt * r, 0, r)
    G.FIELDX, G.FIELDY = dbp_oracle.embed(rx, b, nsymb * nt * r, r), dbp_oracle.embed(ry, b, nsymb * nt * r, r)
    pmx.dbp(fib, flag, step_len=steps, ich=1, decim=r, brf=brf if flag == 'gps-' else None)
    err = rel_l2(G.FIELDX, G.FIELDY, dbp_oracle.embed(tx, b, nsymb * nt * r, r), dbp_oracle.embed(ty, b, nsymb * nt * r, r))
    print('channel dbp exact inverse %s: %d steps, rel_l2 %.3e' % (flag, len(steps), err))
    assert err <= 1e-11


@pytest.mark.gpu
def test_channel_dbp_scalar_path_matches_the_oracle():
    """a scalar 'unique' multiplex of 2^14 samples -- a size full-field DBP has no scalar route for -- channel 3 on 2^10"""
    G = _scalar_unique(512, 32, 3)
    fib = base_fiber(length=8e4, slope=0.057, dphimax=0.02)
    s = fiber_setup(fib, 'g-s-')
    assert not s.isv
    u = G.FIELDX.copy()
    kw = dict(nspan=2, steps_per_span=3)
    pmx.dbp(fib, 'g-s-', gain_db=GAIN_DB, ich=3, decim=16, **kw)
    want = dbp_oracle.dbp_channel_scalar(u, s.betat, s.gam, s.alphalin, s.length, channel_ndfn(3), 16, gain=G16, **kw)
    err = _rel(G.FIELDX, want)
    print('channel dbp scalar parity: rel_l2 %.3e' % err)
    assert G.FIELDY is None or not np.size(G.FIELDY)
    assert err <= 1e-10, err


@pytest.mark.gpu
def test_linear_channel_dbp_is_full_field_dbp_then_the_band_filter(ctx):
    """xi = 0 on the device: single-channel DBP equals full-field DBP followed by a filter plan of the channel's band"""
    gs, s = _setup(512, 32, manakov=True)
    m, r = channel_ndfn(1), 16
    kw = dict(nspan=2, gain_db=GAIN_DB, steps_per_span=3, xi=0.0)
    xs, ys = _batch2(gs)
    cx, cy = _run_device(ctx, s, xs, ys, shift=m, decim=r, **kw)
    fld = _lib.DeviceField(ctx, s.nfft, 1, 2)
    fld.upload(xs, ys)
    plan = dbp_plan(ctx, s, batch=2, **kw)
    plan.execute(fld)
    plan.close()
    H = np.zeros(s.nfft)
    H[dbp_oracle.channel_bins(s.nfft, m, r)] = 1
    band = _lib.Filter(ctx, s.nfft, 1, H, batch=2)
    band.execute(fld)
    band.close()
    fx, fy = fld.download()
    fld.close()
    err = max(rel_l2(cx[b, 0], cy[b, 0], fx[b, 0], fy[b, 0]) for b in range(2))
    assert err <= 1e-12, err


@pytest.mark.gpu
def test_without_dispersion_loss_or_nonlinearity_it_is_the_band_pass(ctx):
    """'----' on a lossless fiber: the output is the ideal band-pass of the input, nothing left outside the band"""
    gs, s = _setup(2048, 32, flag='----', alphadB=0.0)
    assert not s.betat.any() and s.alphalin == 0.0
    m, r = channel_ndfn(3), 16
    xs, ys = _batch2(gs)
    gx, gy = _run_device(ctx, s, xs, ys, shift=m, decim=r, nspan=2, steps_per_span=2)
    b = dbp_oracle.channel_bins(s.nfft, m, r)
    out = np.ones(s.nfft, bool)
    out[b] = False
    for k in range(2):
        err = rel_l2(gx[k, 0], gy[k, 0], dbp_oracle.band_pass(xs[k, 0], b), dbp_oracle.band_pass(ys[k, 0], b))
        spec = np.abs(np.fft.fft(gx[k, 0])) ** 2 + np.abs(np.fft.fft(gy[k, 0])) ** 2
        leak = spec[out].sum() / spec.sum()
        print('band only, realization %d: rel_l2 %.3e, energy outside the band %.3e' % (k, err, leak))
        assert err <= 1e-12 and leak <= 1e-28, (err, leak)


@pytest.mark.gpu
def test_channel_dbp_realizations_are_independent(ctx):
    """single-channel DBP of a batch equals, bit for bit, that of each realization alone (2^20 -> 2^17)"""
    gs, s = _setup(65536, 16, manakov=True)
    xs = np.concatenate([_cols(np.roll(gs.FIELDX, 11 * b, axis=0)) for b in range(3)])
    ys = np.concatenate([_cols(np.roll(gs.FIELDY, -3 * b, axis=0)) for b in range(3)])
    kw = dict(nspan=2, gain_db=GAIN_DB, steps_per_span=2, shift=channel_ndfn(1), decim=8)
    bx, by = _run_device(ctx, s, xs, ys, **kw)
    for b in range(3):
        ox, oy = _run_device(ctx, s, xs[b:b + 1], ys[b:b + 1], **kw)
        assert np.array_equal(ox[0], bx[b]) and np.array_equal(oy[0], by[b]), b


@pytest.mark.gpu
def test_mc_cohmix_with_channel_dbp(ctx):
    """McRunner(receiver='cohmix', compensation='dbp', dbp_params with decim) on a 3-channel 'unique' link runs to the
    end; the field its front-end gets is pmx.dbp(..., ich, decim) of the same received batch"""
    nsymb, nt, nspan, nreal, batch, ich, r = 1 << 11, 16, 2, 4, 2, 3, 8
    ex, ey, sx, sy = synth.pdm_qpsk(nsymb, nt, 3)
    pmx.reset_all(nsymb, nt, 3)
    G = pmx.GSTATE
    G.SYMBOLRATE, G.LAMBDA, G.POWER = 28.0, synth.wdm_lambdas(3, 1550.0, 0.4), np.full(3, 4.0)
    pmx.create_field('unique', ex, ey, {'power': 'average'})
    fib = dict(synth.SMF)
    fib.update(length=8e4, dgd=0.3, nplates=20, manakov='yes')
    setup = fiber_setup(fib, 'gps-', rng=np.random.Generator(np.random.PCG64(0)))
    sym = np.stack([sx[:, ich - 1], sy[:, ich - 1]]).astype(np.uint8)
    x = {'oftype': 'gauss', 'obw': 1.9, 'eftype': 'bessel5', 'ebw': 0.65, 'lopower': 0.0}
    dbpp = dict(steps_per_span=4, decim=r)
    run = mc.McRunner(ctx, setup, G.FIELDX_TX, G.FIELDY_TX, sym, nsymb, nt, nspan, 16.0, 5.0, nreal, batch, receiver='cohmix',
                      dsp_params=dict(mu=1 / 2000, freqavg=200), rx_params=x, ich=ich, pipeline=False,
                      compensation='dbp', dbp_params=dbpp)
    comp, seen = run.rx['cd'], []
    inner = comp.execute

    def spy(field, trace_cap=0):
        before = field.download()
        inner(field)
        seen.append((before, field.download()))
    comp.execute = spy
    try:
        counts, _ = run.run(ase_seed=3)
    finally:
        run.close()
    assert counts.shape == (nreal,) and counts.min() >= 0 and len(seen) == nreal // batch
    errs = []
    for (bx, by), (ax, ay) in seen:
        for b in range(batch):
            G.FIELDX, G.FIELDY = bx[b].T.copy(), by[b].T.copy()
            pmx.dbp(fib, 'gps-', nspan=nspan, gain_db=16.0, steps_per_span=4, ich=ich, decim=r)
            errs.append(rel_l2(ax[b, 0], ay[b, 0], G.FIELDX[:, 0], G.FIELDY[:, 0]))
    print('mc single-channel dbp vs pmx.dbp: rel_l2 %s' % ['%.1e' % e for e in errs])
    assert max(errs) <= 1e-12, errs
