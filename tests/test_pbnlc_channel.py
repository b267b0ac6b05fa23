"""Single-channel PB-NLC (pmx_pb_channel_create, polmux_b200.pbnlc with ich / decim, McRunner with pb_params 'decim'): one
channel of a 'unique' multiplex cut out, compensated at nfft/decim samples with the table of its own dispersion, and
returned to its own bins.

Oracle: tests/pbnlc_channel_oracle.pb_channel -- the full-rate stage oracle on the cropped spectrum, as dbp_oracle.dbp_channel
does it for DBP."""
import ctypes
import importlib
import math
import os
import subprocess

import numpy as np
import pytest

import oracle.fiber_oracle as orc
import dbp_oracle
import pbnlc_channel_oracle as pco
import pbnlc_oracle as po
import polmux_b200 as pmx
from polmux_b200 import _lib, mc, synth
from polmux_b200.fiber import fiber_setup
from polmux_b200.receiver import channel_ndfn
from common import base_fiber, make_tx, rel_l2

pbm = importlib.import_module('polmux_b200.pbnlc')
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GAIN_DB = 16.0


@pytest.fixture
def unique3():
    """a 'unique' multiplex of three 28-GBaud channels at 50 GHz, 256 symbols x 16 samples, in GSTATE"""
    return make_tx(256, 16, nch=3, ftype='unique')


def _desc(**kw):
    """a valid descriptor of the channel at M = nsymb*nt samples, with the fields in kw overridden"""
    nsymb, nt = kw.pop('nsymb', 64), kw.pop('nt', 16)
    d, keep = _lib.make_pb(nsymb, nt, 1, synth.cosroll_pulse(nt, 0.2), pbm.CNLSE, 1.3e-3, 1.0, 1.0, [0, 1], [0, -1],
                           [1.0, 0.5j])
    for k, v in kw.items():
        setattr(d, k, v)
    return d, keep


def _create_rc(d, shift, decim):
    lib = _lib.load()
    band = _lib.make_band(shift, decim)
    h = ctypes.c_void_p()
    rc = lib.pmx_pb_channel_create(None, ctypes.byref(d), ctypes.byref(band), ctypes.byref(h))
    return rc, lib.pmx_last_error(None).decode(), h.value


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_channel_create_validates_before_it_needs_a_context():
    """every refusal comes without a context, with its code and message, and leaves the plan null; a valid request gets
    as far as the missing context"""
    cases = [  # descriptor fields, decim, code, message
        ({}, 3, _lib.PMX_ERR_INVALID, 'decim=3, must be a power of two'),
        ({}, 1, _lib.PMX_ERR_INVALID, 'power of two'),
        ({}, 0, _lib.PMX_ERR_INVALID, 'power of two'),
        (dict(nsymb=16, nt=2), 4, _lib.PMX_ERR_INVALID, 'at least 2^6'),
        (dict(nsymb=1 << 16, nt=16), 32, _lib.PMX_ERR_UNSUPPORTED, '2^24'),
        (dict(nfc=2), 4, _lib.PMX_ERR_UNSUPPORTED, 'nfc=2'),
        (dict(precision=_lib.PMX_F32), 4, _lib.PMX_ERR_UNSUPPORTED, 'FP64 fields only'),
        (dict(nfft=2048), 4, _lib.PMX_ERR_INVALID, 'must equal nfft'),             # what pmx_pb_create rejects
        (dict(npulse=3), 4, _lib.PMX_ERR_INVALID, 'npulse=3'),
        (dict(ncoef=0), 4, _lib.PMX_ERR_INVALID, 'ncoef=0'),
        (dict(batch=0), 4, _lib.PMX_ERR_INVALID, 'batch must be'),
        (dict(xi=float('inf')), 4, _lib.PMX_ERR_INVALID, 'must be finite'),
        ({}, 4, _lib.PMX_ERR_INVALID, 'null ctx'),
    ]
    for kw, decim, code, what in cases:
        d, keep = _desc(**kw)
        rc, msg, h = _create_rc(d, -17, decim)
        assert rc == code and what in msg, (kw, decim, rc, msg)
        assert not h, (kw, decim)


def test_channel_create_prototype_matches_the_header(tmp_path):
    """gcc probe: pmx_pb_channel_create has the type _lib's prototype states"""
    src = tmp_path / 'probe.c'
    src.write_text('#include "polmux_ssfm.h"\n'
                   'int (*f)(pmx_ctx*, const pmx_pb_desc*, const pmx_dbp_band*, pmx_pb_plan**) = pmx_pb_channel_create;\n'
                   'int main(void) { return f == 0; }\n')
    subprocess.run(['gcc', '-Werror', '-c', '-I', os.path.join(ROOT, 'include'), str(src), '-o', str(tmp_path / 'probe.o')],
                   check=True)
    at = _lib.load().pmx_pb_channel_create.argtypes
    assert at == [ctypes.c_void_p, ctypes.POINTER(_lib.PbDesc), ctypes.POINTER(_lib.DbpBand), ctypes.POINTER(ctypes.c_void_p)]
    assert 'pmx_pb_channel_create' in _lib.EXPORTS


def test_python_arguments_are_checked(unique3):
    fib = base_fiber()
    with pytest.raises(ValueError, match='needs decim'):
        pmx.pbnlc(fib, 'g-s-', 2, ich=1)                                       # ich without decim
    with pytest.raises(ValueError, match='needs the channel ich'):
        pmx.pbnlc(fib, 'g-s-', 2, decim=8)                                     # decim without ich
    with pytest.raises(ValueError, match='does not exist'):
        pmx.pbnlc(fib, 'g-s-', 2, ich=4, decim=8)
    with pytest.raises(ValueError, match='power of two'):
        pmx.pbnlc(fib, 'g-s-', 2, ich=1, decim=3)
    with pytest.raises(ValueError, match='must divide nt'):
        pmx.pbnlc(fib, 'g-s-', 2, ich=1, decim=32)
    s = fiber_setup(fib, 'g-s-')
    with pytest.raises(ValueError, match='needs decim'):
        pbm.pb_plan(None, s, 2, shift=5)
    make_tx(256, 16, nch=3, ftype='sepfields')                                 # nfc = 3
    with pytest.raises(ValueError, match="one column"):
        pmx.pbnlc(fib, 'g-s-', 2, ich=1, decim=8)
    with pytest.raises(ValueError, match='nfc=3'):
        pbm.pb_plan(None, fiber_setup(fib, 'g-s-'), 2, shift=0, decim=8)


def test_without_decim_a_multiplex_is_still_refused(unique3):
    with pytest.raises(ValueError, match='one channel'):
        pmx.pbnlc(base_fiber(), 'g-s-', 2)


@pytest.mark.skipif(_lib.load().pmx_device_count() > 0, reason='a GPU is present')
def test_channel_pbnlc_has_no_cpu_fallback(unique3):
    with pytest.raises(_lib.PolmuxError):
        pmx.pbnlc(base_fiber(), 'g-s-', 2, K=2, ich=1, decim=8)


def _tables(slope):
    """the tables (K = 8, 3 spans) of the centre and both edge channels of nine at 2^15 samples, decim 8"""
    make_tx(1024, 32, nch=9)
    fib = base_fiber(slope=slope)
    s = fiber_setup(fib, 'g-s-')
    p = pbm.channel_pulse(32, 8, s.nfft)
    return s, [pbm.pb_coefficients(pbm.channel_setup(s, channel_ndfn(i), 8), 3, p, 8, nt=4, nquad=8)[2] for i in (5, 1, 9)]


def test_channel_table_differs_from_the_centre_only_with_a_dispersion_slope():
    """b30 = 0: an edge channel's table is the centre channel's (the group delay and phase of a channel cancel in the
    triplet products); with the fibre's dispersion slope it is not"""
    s, (c, e1, e9) = _tables(-2 * synth.SMF['disp'] / synth.SMF['lambda'])             # slope that makes b30 = 0
    assert s.scalars['b30'] == 0.0
    c00 = abs(c[c.size // 2])
    d0 = max(np.abs(e1 - c).max(), np.abs(e9 - c).max()) / c00
    s, (c, e1, e9) = _tables(0.057)
    assert s.scalars['b30'] != 0.0
    d1 = min(np.abs(e1 - c).max(), np.abs(e9 - c).max()) / abs(c[c.size // 2])
    print('edge vs centre table / |C[0,0]|: b30 = 0 %.2e, b30 != 0 %.2e' % (d0, d1))
    assert d0 <= 1e-12 and d1 > 1e-6


def test_channel_pulse_is_the_band_passed_transmit_pulse():
    """the default pulse at nt/decim: even, 16*nt/decim samples, and the decimated band-pass of the transmit pulse on the
    samples it keeps"""
    nt, r, N = 16, 4, 1 << 12
    p = pbm.channel_pulse(nt, r, N)
    assert p.size == 16 * nt // r and p.dtype == np.float64
    u = po.pulse_at(synth.cosroll_pulse(nt, 0.2), nt, N, 0)
    v = dbp_oracle.crop(u, dbp_oracle.channel_bins(N, 0, r), r)
    assert np.abs(p - v[(np.arange(p.size) - p.size // 2) % (N // r)].real).max() <= 1e-15


def test_oracle_at_xi0_is_the_band_pass(unique3):
    """xi = 0: pb_channel is the crop-and-embed band-pass; on a field already on the channel's bins it returns the field"""
    gs = unique3
    N, r, m = gs.FIELDX.shape[0], 4, channel_ndfn(1)
    b = dbp_oracle.channel_bins(N, m, r)
    p = pbm.channel_pulse(16, r, N)
    ux, uy = gs.FIELDX[:, 0], gs.FIELDY[:, 0]
    ox, oy, _, _ = pco.pb_channel(ux, uy, p, 4, [0], [0], [1.0], pbm.CNLSE, 1.3e-3, 1.0, 0.0, m, r)
    assert rel_l2(ox, oy, dbp_oracle.band_pass(ux, b), dbp_oracle.band_pass(uy, b)) <= 1e-13
    bx, by = dbp_oracle.band_pass(ux, b), dbp_oracle.band_pass(uy, b)
    ox, oy, _, _ = pco.pb_channel(bx, by, p, 4, [0], [0], [1.0], pbm.CNLSE, 1.3e-3, 1.0, 0.0, m, r)
    assert rel_l2(ox, oy, bx, by) <= 1e-13


# ---------------------------------------------------------------------------------------------------------------- GPU
def _batch(gs, batch):
    """batch different realizations of the multiplex: shifted in time, the x polarization turned -> (x, y) [batch][1][nfft]"""
    xs = np.stack([np.roll(gs.FIELDX[:, 0], 7 * b) * np.exp(0.3j * b) for b in range(batch)])[:, None]
    ys = np.stack([np.roll(gs.FIELDY[:, 0], -5 * b) for b in range(batch)])[:, None]
    return np.ascontiguousarray(xs), np.ascontiguousarray(ys)


def _rel(a, b):
    return float(np.linalg.norm(np.ravel(a) - np.ravel(b)) / np.linalg.norm(np.ravel(b)))


def _plan(ctx, s, nt, r, m, K, batch, xi):
    """the channel plan of 2 spans with the table of channel_setup -> (plan, pulse, table, weights, gamma, scale)"""
    p = pbm.channel_pulse(nt, r, s.nfft)
    tab = pbm.pb_coefficients(pbm.channel_setup(s, m, r), 2, p, K, nt=nt // r, nquad=8)
    w, gam = pbm.model_weights(s)
    plan = pbm.pb_plan(ctx, s, 2, GAIN_DB, xi=xi, K=K, batch=batch, nt=nt, coefs=tab, shift=m, decim=r)
    return plan, p, tab, w, gam, pbm.scale_factor(s, 2, GAIN_DB)


CHANNEL = [  # nsymb, nt, decim, nch, ich, batch, manakov, K
    (512, 16, 4, 3, 1, 16, False, 16),          # 2^13 transposed -> 2^11 natural, edge of 3
    (256, 32, 4, 9, 5, 1, True, 0),             # 2^13 -> 2^11, centre of 9
    (2048, 32, 16, 9, 9, 16, True, 32),         # 2^16 -> 2^12, edge of 9
    (4096, 16, 16, 3, 2, 1, False, 32),         # 2^16 -> 2^12, centre of 3, one sample per symbol
    (65536, 16, 16, 3, 3, 1, False, 16),        # 2^20 -> 2^16, edge of 3
    (32768, 32, 16, 9, 1, 16, True, 0),         # 2^20 -> 2^16, edge of 9
]


@pytest.mark.gpu
@pytest.mark.parametrize('case', CHANNEL, ids=lambda c: '2^%d-r%d-nch%d-ch%d-b%d-%s-K%d' % (
    int(math.log2(c[0] * c[1])), c[2], c[3], c[4], c[5], 'man' if c[6] else 'cnlse', c[7]))
def test_channel_stage_matches_the_oracle(ctx, case):
    """projected symbols and triplet sum (<= 1e-12) and the corrected field (<= 1e-10) against pb_channel, every
    realization its own field, the bounds of the full-rate stage"""
    nsymb, nt, r, nch, ich, batch, manakov, K = case
    gs = make_tx(nsymb, nt, nch=nch, ftype='unique', pavg_mw=4.0)
    s = fiber_setup(base_fiber(slope=0.057), 'g-s-')
    s.manakov = manakov
    m = channel_ndfn(ich) if nch > 1 else 0
    xs, ys = _batch(gs, batch)
    plan, p, (mm, nn, C), w, gam, scale = _plan(ctx, s, nt, r, m, K, batch, 0.8)
    fld = _lib.DeviceField(ctx, s.nfft, 1, batch)
    fld.upload(xs, ys)
    plan.execute(fld)
    A, D = plan.symbols()
    ox, oy = fld.download()
    plan.close()
    fld.close()
    assert A.shape == (batch, 2, nsymb)
    bins = dbp_oracle.channel_bins(s.nfft, m, r)
    a_ref, u_dev, u_ref = [], [], []
    for b in range(batch):
        rx, ry, ab, _ = pco.pb_channel(xs[b, 0], ys[b, 0], p, nt // r, mm, nn, C, w, gam, scale, 0.8, m, r)
        a_ref.append(ab)
        bx, by = dbp_oracle.band_pass(xs[b, 0], bins), dbp_oracle.band_pass(ys[b, 0], bins)
        u_dev.append(np.concatenate([ox[b, 0] - bx, oy[b, 0] - by]))
        u_ref.append(np.concatenate([rx - bx, ry - by]))
    a_ref = np.stack(a_ref)
    eA, eD = _rel(A, a_ref), _rel(D, po.triplets(A, mm, nn, C, w, gam, scale))
    eF, eU = _rel(D, po.triplets(a_ref, mm, nn, C, w, gam, scale)), _rel(np.array(u_dev), np.array(u_ref))
    print('pb channel %s: ncoef %d  A %.2e  Delta %.2e  Delta(oracle A) %.2e  correction %.2e'
          % (case, len(C), eA, eD, eF, eU))
    assert eA <= 1e-12 and eD <= 1e-12 and eF <= 1e-10 and eU <= 1e-10


@pytest.mark.gpu
def test_channel_stage_is_deterministic_and_xi0_is_the_band_pass(ctx):
    """two executions give the same bits; xi = 0 gives the oracle's band-pass of the input and launches no PB kernel (three
    launches fewer than xi = 1: project, triplets, apply)"""
    nsymb, nt, r, batch = 4096, 16, 8, 4
    gs = make_tx(nsymb, nt, nch=3, ftype='unique', pavg_mw=4.0)
    s = fiber_setup(base_fiber(), 'g-s-')
    m = channel_ndfn(1)
    xs, ys = _batch(gs, batch)
    fld = _lib.DeviceField(ctx, s.nfft, 1, batch)
    outs, launches = [], []
    for xi in (1.0, 1.0, 0.0):
        plan = _plan(ctx, s, nt, r, m, 16, batch, xi)[0]
        fld.upload(xs, ys)
        n0 = ctx.launches
        plan.execute(fld)
        launches.append(ctx.launches - n0)
        plan.close()
        outs.append(fld.download())
    fld.close()
    assert np.array_equal(outs[0][0].view(np.uint64), outs[1][0].view(np.uint64))
    assert np.array_equal(outs[0][1].view(np.uint64), outs[1][1].view(np.uint64))
    assert launches[0] == launches[1] == launches[2] + 3, launches
    bins = dbp_oracle.channel_bins(s.nfft, m, r)
    err = max(rel_l2(outs[2][0][b, 0], outs[2][1][b, 0], dbp_oracle.band_pass(xs[b, 0], bins),
                     dbp_oracle.band_pass(ys[b, 0], bins)) for b in range(batch))
    print('xi = 0 against the band-pass: rel_l2 %.2e, launches %s' % (err, launches))
    assert err <= 1e-13


@pytest.mark.gpu
def test_channel_stage_refuses_a_field_it_was_not_made_for(ctx):
    """a plan for 2^12 samples (decim 4) refuses other lengths and batches, and more than one column"""
    make_tx(256, 16)
    plan = pbm.pb_plan(ctx, fiber_setup(base_fiber(), 'g-s-'), 2, GAIN_DB, K=2, nt=16, coefs=([0], [0], [1.0]), shift=0, decim=4)
    for kw, what in ((dict(nfft=1 << 11, nfc=1, batch=1), 'nfft=2048'), (dict(nfft=1 << 12, nfc=1, batch=2), 'batch 2'),
                     (dict(nfft=1 << 12, nfc=2, batch=1), 'nfc=2')):
        fld = _lib.DeviceField(ctx, **kw)
        with pytest.raises(_lib.PolmuxError, match=what) as e:
            plan.execute(fld)
        assert e.value.code == (_lib.PMX_ERR_UNSUPPORTED if kw['nfc'] > 1 else _lib.PMX_ERR_INVALID)
        fld.close()
    plan.close()


def _unequal_multiplex(nsymb, nt, powers):
    """GSTATE <- a 'unique' multiplex of len(powers) channels at 50 GHz with those launch powers [mW]; -> oracle GState"""
    nch = len(powers)
    ex, ey, sx, sy = synth.pdm_qpsk(nsymb, nt, nch)
    lams = synth.wdm_lambdas(nch, 1550.0, 0.4)
    gs = orc.reset_all(nsymb, nt, nch)
    gs.SYMBOLRATE, gs.LAMBDA, gs.POWER = 28.0, lams.copy(), np.array(powers, dtype=np.float64)
    orc.create_field(gs, 'unique', ex, ey, power_average=True)
    pmx.reset_all(nsymb, nt, nch)
    G = pmx.GSTATE
    G.SYMBOLRATE, G.LAMBDA, G.POWER = 28.0, lams.copy(), np.array(powers, dtype=np.float64)
    pmx.create_field('unique', ex, ey, {'power': 'average'})
    return gs, sx, sy


@pytest.mark.gpu
def test_channel_pbnlc_lowers_the_residual_below_cd_only():
    """three channels, 5 x 80 km, noise-free, the centre one at 4 mW between neighbours at 0.5 mW, so that its own
    nonlinear distortion dominates the cross-phase modulation no single-channel method undoes: the symbol-centre residual
    of the centre channel against its Tx (band-passed like the field) after CD + band-pass, single-channel PB-NLC and
    single-channel DBP at one step per span, all at decim 16 (two samples per symbol)"""
    nsymb, nt, nspan, r, ich = 512, 32, 5, 16, 2
    gs, _, _ = _unequal_multiplex(nsymb, nt, [0.5, 4.0, 0.5])
    fib = base_fiber(dphimax=1e-3)
    s = fiber_setup(fib, 'g-s-')
    g = math.exp(s.alphalin * s.length)
    ux, uy = gs.FIELDX.copy(), gs.FIELDY.copy()
    for _ in range(nspan):
        _, _, ux, uy, _, _ = orc.matrix_ssfm(ux, uy, s.betat, s.db1, s.dzmaxt, s.dphimaxt, s.gam, s.alphalin, 1, s.length, 1,
                                             'no', s.fls, s.brf)
        ux, uy = ux * math.sqrt(g), uy * math.sqrt(g)
    gain_db = 10 * math.log10(g)
    m = channel_ndfn(ich)
    bins = dbp_oracle.channel_bins(s.nfft, m, r)
    tx, ty = dbp_oracle.band_pass(gs.FIELDX[:, 0], bins)[::nt], dbp_oracle.band_pass(gs.FIELDY[:, 0], bins)[::nt]
    G = pmx.GSTATE
    res = {}
    for what in ('cd', 'pbnlc', 'dbp'):
        G.FIELDX, G.FIELDY = ux.copy(), uy.copy()
        if what == 'cd':
            pmx.pbnlc(fib, 'g-s-', nspan, gain_db, xi=0.0, K=0, ich=ich, decim=r)
        elif what == 'pbnlc':
            pmx.pbnlc(fib, 'g-s-', nspan, gain_db, xi=1.0, K=32, ich=ich, decim=r)
        else:
            pmx.dbp(fib, 'g-s-', nspan, gain_db, steps_per_span=1, ich=ich, decim=r)
        ox, oy = np.asarray(G.FIELDX)[::nt, 0], np.asarray(G.FIELDY)[::nt, 0]
        res[what] = math.sqrt((np.sum(np.abs(ox - tx) ** 2) + np.sum(np.abs(oy - ty) ** 2))
                              / (np.sum(np.abs(tx) ** 2) + np.sum(np.abs(ty) ** 2)))
    print('centre channel of three, symbol-centre residual vs Tx: CD + band-pass %.4f, single-channel PB-NLC (K=32) %.4f, '
          'single-channel DBP 1 step/span %.4f' % (res['cd'], res['pbnlc'], res['dbp']))
    assert res['pbnlc'] < 0.9 * res['cd']


def _mc_link(nsymb, nt, powers, dgd):
    gs, sx, sy = _unequal_multiplex(nsymb, nt, powers)
    fib = dict(synth.SMF)
    fib.update(length=8e4, dgd=dgd, nplates=20, manakov='yes')
    setup = fiber_setup(fib, 'gps-', rng=np.random.Generator(np.random.PCG64(0)))
    return fib, setup, sx, sy


COHMIX = {'oftype': 'gauss', 'obw': 1.9, 'eftype': 'bessel5', 'ebw': 0.65, 'lopower': 0.0}


@pytest.mark.gpu
def test_mc_cohmix_with_channel_pbnlc(ctx):
    """McRunner(receiver='cohmix', compensation='pbnlc', pb_params with decim) on a 3-channel 'unique' link runs to the end,
    and the field its front-end gets is pmx.pbnlc(..., ich, decim) of the same received batch"""
    nsymb, nt, nspan, nreal, batch, ich, r = 1 << 11, 16, 2, 4, 2, 3, 8
    fib, setup, sx, sy = _mc_link(nsymb, nt, [4.0, 4.0, 4.0], 0.3)
    G = pmx.GSTATE
    sym = np.stack([sx[:, ich - 1], sy[:, ich - 1]]).astype(np.uint8)
    run = mc.McRunner(ctx, setup, G.FIELDX_TX, G.FIELDY_TX, sym, nsymb, nt, nspan, GAIN_DB, 5.0, nreal, batch,
                      receiver='cohmix', dsp_params=dict(mu=1 / 2000, freqavg=200), rx_params=COHMIX, ich=ich,
                      pipeline=False, compensation='pbnlc', pb_params=dict(K=8, decim=r))
    cd, pb, seen = run.rx['cd'], run.rx['pb'], []
    cd_exec, pb_exec = cd.execute, pb.execute

    def spy_cd(field, *a, **k):
        seen.append([field.download()])
        cd_exec(field, *a, **k)

    def spy_pb(field):
        pb_exec(field)
        seen[-1].append(field.download())
    cd.execute, pb.execute = spy_cd, spy_pb
    try:
        counts, _ = run.run(ase_seed=3)
    finally:
        run.close()
    assert counts.shape == (nreal,) and counts.min() >= 0 and len(seen) == nreal // batch
    errs = []
    for (bx, by), (ax, ay) in seen:
        for b in range(batch):
            G.FIELDX, G.FIELDY = bx[b].T.copy(), by[b].T.copy()
            pmx.pbnlc(fib, 'gps-', nspan, GAIN_DB, K=8, ich=ich, decim=r)
            errs.append(rel_l2(ax[b, 0], ay[b, 0], G.FIELDX[:, 0], G.FIELDY[:, 0]))
    print('mc single-channel pbnlc vs pmx.pbnlc: rel_l2 %s' % ['%.1e' % e for e in errs])
    assert max(errs) <= 1e-12, errs


@pytest.mark.gpu
def test_mc_cohmix_channel_pbnlc_counts_fewer_errors_than_cd(ctx):
    """the centre channel of three, 10 x 80 km, at 12 mW between neighbours at 2 mW: single-channel PB-NLC (decim 8,
    K = 32) counts fewer errors than 'cd' on the same realizations, and two runs count the same"""
    nsymb, nt, nspan, nreal, batch, ich, r = 1 << 12, 16, 10, 16, 8, 2, 8
    fib, setup, sx, sy = _mc_link(nsymb, nt, [2.0, 12.0, 2.0], 0.1)
    G = pmx.GSTATE
    sym = np.stack([sx[:, ich - 1], sy[:, ich - 1]]).astype(np.uint8)
    out = {}
    for what, comp, pb in (('cd', 'cd', None), ('pb', 'pbnlc', dict(K=32, decim=r))):
        run = mc.McRunner(ctx, setup, G.FIELDX_TX, G.FIELDY_TX, sym, nsymb, nt, nspan, GAIN_DB, 5.0, nreal, batch,
                          receiver='cohmix', dsp_params=dict(mu=1 / 2000, freqavg=200), rx_params=COHMIX, ich=ich,
                          compensation=comp, pb_params=pb)
        try:
            out[what] = [run.run(ase_seed=3)[0] for _ in range(2 if what == 'pb' else 1)]
        finally:
            run.close()
    print('mc cohmix centre of three: errors cd %d, single-channel pbnlc %d'
          % (out['cd'][0].sum(), out['pb'][0].sum()))
    assert np.array_equal(out['pb'][0], out['pb'][1])
    assert out['cd'][0].sum() > 0
    assert out['pb'][0].sum() < out['cd'][0].sum()
