"""XPM-aware single-channel PB-NLC (pbnlc.xpm_coefficients, pmx_pb_xpm_create, pb_plan / pmx.pbnlc with xpm, McRunner with
pb_params 'xpm'): the channel's cross-phase modulation compensated from the neighbours' projected symbols.

Oracle: tests/pbnlc_xpm_oracle.py -- the weights from the forward oracle's nonlinear step, the direct overlap integral,
and the stage (crop, project, SPM and XPM triplets, apply, embed)."""
import ctypes
import importlib
import math
import os
import subprocess

import numpy as np
import pytest

import oracle.fiber_oracle as orc
import dbp_oracle
import pbnlc_oracle as po
import pbnlc_xpm_oracle as pxo
import polmux_b200 as pmx
from polmux_b200 import _lib, mc, synth
from polmux_b200.fiber import fiber_setup
from polmux_b200.receiver import channel_ndfn
from common import base_fiber, make_tx

pbm = importlib.import_module('polmux_b200.pbnlc')
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GAIN_DB = 16.0


def _rel(a, b):
    return float(np.linalg.norm(np.ravel(a) - np.ravel(b)) / np.linalg.norm(np.ravel(b)))


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize('manakov', [False, True])
def test_weights_are_the_first_order_step_on_two_tones(manakov):
    """u = A + B*exp(2*pi*i*q*t/N): the part of the nonlinear step's first-order term at the COI's frequency (bin 0) that
    the interferer adds is -j*gam*(w1 Ax|Bx|^2 + w2 Ax|By|^2 + w3 Ay Bx conj(By) + w4 Ay By conj(Bx)) (x <-> y)"""
    N, q, gam = 16, 3, 1.3e-3
    rng = np.random.default_rng(5)
    A = rng.standard_normal(2) + 1j * rng.standard_normal(2)
    B = rng.standard_normal(2) + 1j * rng.standard_normal(2)
    e = np.exp(2j * np.pi * q * np.arange(N) / N)
    h = 1e-4 / gam
    f1 = pxo.first_order(A[0] + B[0] * e, A[1] + B[1] * e, manakov, gam, h)
    f0 = pxo.first_order(np.full(N, A[0]), np.full(N, A[1]), manakov, gam, h)
    meas = np.array([np.mean(f1[i]) - np.mean(f0[i]) for i in range(2)])
    w1, w2, w3, w4 = pbm.MANAKOV_XPM if manakov else pbm.CNLSE_XPM
    ax, ay, bx, by = A[0], A[1], B[0], B[1]
    pred = -1j * gam * np.array([w1 * ax * abs(bx) ** 2 + w2 * ax * abs(by) ** 2 + w3 * ay * bx * np.conj(by)
                                 + w4 * ay * by * np.conj(bx),
                                 w1 * ay * abs(by) ** 2 + w2 * ay * abs(bx) ** 2 + w3 * ax * by * np.conj(bx)
                                 + w4 * ax * bx * np.conj(by)])
    err = np.abs(meas - pred).max() / np.abs(pred).max()
    print('two-tone XPM weights (manakov=%s): residual %.1e' % (manakov, err))
    assert err <= 1e-12


def _small():
    """two channels at 50 GHz, 64 symbols x 16 samples, decim 4; -> (setup, COI shift, interferer shift, pulse)"""
    make_tx(64, 16, nch=2)
    s = fiber_setup(base_fiber(length=4e4, slope=0.057), 'g-s-')
    return s, channel_ndfn(1), channel_ndfn(2), pbm.channel_pulse(16, 4, s.nfft)


def test_fast_table_equals_the_direct_overlap_integral():
    """the FFT form of xpm_coefficients against the term-by-term integral of the oracle, both on the whole block; the
    table is D[-m,n] = conj(D[m,n]) exactly and has no m <-> n symmetry"""
    s, m0, m1, p = _small()
    K, Kn = 2, 6
    m, n, D = pbm.xpm_coefficients(s, 2, m0, m1, 4, p, K, Kn, nt=16, nquad=4, window=64)
    Dd = pxo.coefficients_direct(s.betat[:, 0], m0, m1, 4, 16, s.length, s.alphalin, 2, p, K, Kn, 4, 4)
    Df = D.reshape(2 * K + 1, 2 * Kn + 1)
    assert np.array_equal(m.reshape(Df.shape)[:, 0], np.arange(-K, K + 1))
    assert np.array_equal(n.reshape(Df.shape)[0], np.arange(-Kn, Kn + 1))
    err = np.abs(Df - Dd).max() / np.abs(Dd).max()
    asym = np.abs(Df[:, Kn - K:Kn + K + 1] - Df[:, Kn - K:Kn + K + 1].T).max() / np.abs(Dd).max()
    print('XPM table: FFT form vs direct %.1e of max|D|; |D[m,n] - D[n,m]| up to %.2f of max|D|' % (err, asym))
    assert err <= 1e-12
    assert np.array_equal(Df[::-1], np.conj(Df))
    assert asym > 1e-3


def test_table_does_not_alias():
    """doubling the table's rate changes the table by <= 1e-10 of max|D| (measured 2e-16), while at nt/decim samples per
    symbol the four-pulse products alias (3e-2).  Doubling the default window changes it by 1.1e-7 of max|D|, and the
    change falls 4x with every further doubling (2.7e-8, 6.9e-9, 1.7e-9 from 512 to 2048 symbols): the band-limited pulse
    carries the sinc tails of the band's edge, which wrap on a circular window; only the whole block removes them."""
    make_tx(2048, 16, nch=3)
    s = fiber_setup(base_fiber(), 'g-s-')
    m0, m1 = channel_ndfn(2), channel_ndfn(3)
    p = pbm.channel_pulse(16, 8, s.nfft)
    kw = dict(K=4, Kn=40, nt=16, nquad=8)
    W = pbm.default_xpm_window(s, 3, m0, m1, 8, p, 16, 4, 40)
    base = pbm.xpm_coefficients(s, 3, m0, m1, 8, p, **kw)[2]
    wide = pbm.xpm_coefficients(s, 3, m0, m1, 8, p, window=2 * W, **kw)[2]
    fine = pbm.xpm_coefficients(s, 3, m0, m1, 8, p, up=8, **kw)[2]
    coarse = pbm.xpm_coefficients(s, 3, m0, m1, 8, p, up=1, **kw)[2]
    big = np.abs(base).max()
    dw, du, d1 = (np.abs(x - base).max() / big for x in (wide, fine, coarse))
    print('XPM table (window %d): doubled window %.1e, doubled rate %.1e, at nt/decim (no zero-padding) %.1e of max|D|'
          % (W, dw, du, d1))
    assert W < 2048 and dw <= 2e-7 and du <= 1e-10
    assert d1 > 1e-6                          # the products alias at two samples per symbol


def _two_channel_link(pmw, nspan, neighbour, nsymb=256, nt=8):
    """the COI (channel 1) with or without a 50 GHz neighbour (channel 2), both at pmw, noise-free oracle link -> (Tx (x, y),
    CD-compensated Rx (x, y), setup)"""
    ex, ey, _, _ = synth.pdm_qpsk(nsymb, nt, 2)
    lams = synth.wdm_lambdas(2, 1550.0, 0.4)
    gs = orc.reset_all(nsymb, nt, 2)
    gs.SYMBOLRATE, gs.LAMBDA, gs.POWER = 28.0, lams.copy(), np.array([pmw, pmw if neighbour else 0.0])
    orc.create_field(gs, 'unique', ex, ey, power_average=True)
    pmx.reset_all(nsymb, nt, 2)
    G = pmx.GSTATE
    G.SYMBOLRATE, G.LAMBDA, G.POWER = 28.0, lams.copy(), gs.POWER.copy()
    pmx.create_field('unique', ex, ey, {'power': 'average'})
    s = fiber_setup(base_fiber(dphimax=1e-3), 'g-s-')
    g = math.exp(s.alphalin * s.length)
    ux, uy = gs.FIELDX.copy(), gs.FIELDY.copy()
    for _ in range(nspan):
        _, _, ux, uy, _, _ = orc.matrix_ssfm(ux, uy, s.betat, s.db1, s.dzmaxt, s.dphimaxt, s.gam, s.alphalin, 1, s.length, 1,
                                             'no', s.fls, s.brf)
        ux, uy = ux * math.sqrt(g), uy * math.sqrt(g)
    bt = s.betat * (s.length * nspan)
    return (gs.FIELDX, gs.FIELDY), (orc.lin_step(-bt, ux), orc.lin_step(-bt, uy)), s


def _xpm_mismatch(pmw, K=16, nspan=3, nt=8, r=4):
    """|XPM_meas - XPM_pred| / |XPM_meas| of the COI's projected symbols: measured, with the neighbour minus without it;
    predicted, the XPM triplets of the table on the Tx symbols"""
    tx, rx, s = _two_channel_link(pmw, nspan, True)
    tx0, rx0, _ = _two_channel_link(pmw, nspan, False)
    m0, m1 = channel_ndfn(1), channel_ndfn(2)
    p = pbm.channel_pulse(nt, r, s.nfft)
    a = lambda u, sh: pxo.channel_symbols(*u, p, nt // r, sh, r)
    a_tx, b_tx = a(tx, m0), a(tx, m1)
    # (each against its own Tx: the neighbour's linear leak into the COI's band cancels)
    a_with, a_without = a(rx, m0) - a_tx, a(rx0, m0) - a(tx0, m0)
    m, n, D = pbm.xpm_coefficients(s, nspan, m0, m1, r, p, K, nt=nt)
    w, gam = pbm.xpm_weights(s)
    d_meas, d_pred = a_with - a_without, pxo.xpm_triplets(a_tx, b_tx, m, n, D, w, gam)
    return np.linalg.norm(d_meas - d_pred) / np.linalg.norm(d_meas)


def test_table_is_the_links_first_order_xpm_term():
    """COI and one 50 GHz neighbour (no four-wave mixing lands on the COI), 3 x 80 km, no noise, dphimax 1e-3, K = 16: the
    XPM the forward oracle gives the COI's projected symbols (with the neighbour minus without) against the XPM triplets of
    the table on the Tx symbols (each run against its own Tx, so that the neighbour's linear leak into the COI's band
    cancels).  Measured: 0.343 / 0.140 / 0.119 at 2 / 0.5 / 0.125 mW per channel.  The floor of about 12 % is the part of
    the first-order term the triplet form leaves out (indices with i + j - l != k); above it the mismatch is second order:
    once the floor is taken out (in quadrature) it shrinks 4.3x when the power is divided by 4."""
    e = [_xpm_mismatch(p) for p in (2.0, 0.5, 0.125)]
    print('first-order XPM mismatch at 2 / 0.5 / 0.125 mW: %s' % ['%.4f' % v for v in e])
    assert e[2] < FLOOR
    hi, lo = math.sqrt(e[0] ** 2 - e[2] ** 2), math.sqrt(max(e[1] ** 2 - e[2] ** 2, 0.0))
    assert 3.0 < hi / lo < 5.5, (e, hi / lo)


FLOOR = 0.14


def _desc(**kw):
    """valid descriptors of a channel at M = 64 x 16 samples, decim 4, and two interferers, with fields overridden"""
    d, keep = _lib.make_pb(64, 16, 1, synth.cosroll_pulse(16, 0.2), pbm.CNLSE, 1.3e-3, 1.0, 1.0, [0], [0], [1.0])
    xd = _lib.make_pb_xpm(kw.pop('shifts', [100, -100]), kw.pop('tables', [([0, 1], [0, -3], [1.0, 0.5j])] * 2),
                          kw.pop('weights', pbm.CNLSE_XPM))
    for k, v in kw.items():
        setattr(d, k, v)
    return (d, keep), xd


def _create_rc(desc_keep, xd, shift=0, decim=4):
    lib = _lib.load()
    band = _lib.make_band(shift, decim)
    h = ctypes.c_void_p()
    rc = lib.pmx_pb_xpm_create(None, ctypes.byref(desc_keep[0]), ctypes.byref(band), ctypes.byref(xd[0]), ctypes.byref(h))
    return rc, lib.pmx_last_error(None).decode(), h.value


def test_xpm_create_validates_before_it_needs_a_context():
    """every refusal comes without a context, with its code and message, and leaves the plan null; a valid request gets
    as far as the missing context"""
    one = ([0], [0], [1.0])
    cases = [  # make_pb overrides / xpm keywords, decim, code, message
        (dict(shifts=[], tables=[]), 4, _lib.PMX_ERR_INVALID, 'nint=0'),
        (dict(shifts=list(range(1, 10)), tables=[one] * 9), 4, _lib.PMX_ERR_INVALID, 'nint=9'),
        (dict(shifts=[0], tables=[one]), 4, _lib.PMX_ERR_INVALID, "the channel's own shift"),
        (dict(shifts=[4096 + 0, 7], tables=[one] * 2), 4, _lib.PMX_ERR_INVALID, "the channel's own shift"),   # mod N
        (dict(shifts=[7, 7 - 4096]), 4, _lib.PMX_ERR_INVALID, 'the same shift'),
        (dict(tables=[([0], [0], [1.0]), ([], [], [])]), 4, _lib.PMX_ERR_INVALID, 'ncoef=0'),
        (dict(tables=[([129], [0], [1.0]), one]), 4, _lib.PMX_ERR_INVALID, '|m| at most 128'),
        (dict(tables=[one, ([0], [1025], [1.0])]), 4, _lib.PMX_ERR_INVALID, '|n| at most 1024'),
        (dict(tables=[one, ([0], [-1024], [float('nan')])]), 4, _lib.PMX_ERR_INVALID, 'coefficient 1 is not finite'),
        (dict(weights=(2, 1, float('inf'), 0)), 4, _lib.PMX_ERR_INVALID, 'weight 2'),
        (dict(precision=_lib.PMX_F32), 4, _lib.PMX_ERR_UNSUPPORTED, 'FP64 fields only'),   # pmx_pb_channel_create's
        (dict(nfc=2), 4, _lib.PMX_ERR_UNSUPPORTED, 'nfc=2'),
        ({}, 3, _lib.PMX_ERR_INVALID, 'decim=3'),
        (dict(npulse=3), 4, _lib.PMX_ERR_INVALID, 'npulse=3'),
        ({}, 4, _lib.PMX_ERR_INVALID, 'null ctx'),
    ]
    for kw, decim, code, what in cases:
        dk, xd = _desc(**kw)
        rc, msg, h = _create_rc(dk, xd, 0, decim)
        assert rc == code and what in msg, (kw, decim, rc, msg)
        assert not h, (kw, decim)
    dk, xd = _desc()
    xd[0].ncoef = None
    assert _create_rc(dk, xd)[:2] == (_lib.PMX_ERR_INVALID, 'pmx_pb_xpm_create: null interferer list')


def test_xpm_desc_and_prototypes_match_the_header(tmp_path):
    """a gcc probe against the header: pmx_pb_xpm_desc's size and offsets equal the ctypes mirror, the limits equal
    _lib's, and the prototypes compile with the argument types the binding passes"""
    cls = _lib.PbXpmDesc
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "polmux_ssfm.h"',
             'static int (*f1)(pmx_ctx*, const pmx_pb_desc*, const pmx_dbp_band*, const pmx_pb_xpm_desc*, pmx_pb_plan**) = '
             'pmx_pb_xpm_create;', 'static int (*f2)(pmx_pb_plan*, int32_t, double*) = pmx_pb_xpm_symbols;',
             'int main(void){', 'printf("size %zu\\n", sizeof(pmx_pb_xpm_desc));',
             'printf("maxint %d\\n", PMX_PB_XPM_MAX_INT);', 'printf("maxn %d\\n", PMX_PB_XPM_MAX_N);']
    for fname, _ in cls._fields_:
        lines.append('printf("%s %%zu\\n", offsetof(pmx_pb_xpm_desc, %s));' % (fname, fname))
    lines.append('return f1 == 0 || f2 == 0;}')
    src = tmp_path / 'probe.c'
    src.write_text('\n'.join(lines))
    exe = tmp_path / 'probe'
    subprocess.run(['gcc', '-Werror', '-I', os.path.join(ROOT, 'include'), str(src), '-o', str(exe),
                    '-Wl,--unresolved-symbols=ignore-all'], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True).stdout.splitlines())
    assert int(out['size']) == ctypes.sizeof(cls)
    for fname, _ in cls._fields_:
        assert int(out[fname]) == getattr(cls, fname).offset, fname
    assert int(out['maxint']) == _lib.PB_XPM_MAX_INT and int(out['maxn']) == _lib.PB_XPM_MAX_N
    lib = _lib.load()
    assert lib.pmx_pb_xpm_create.argtypes == [ctypes.c_void_p, ctypes.POINTER(_lib.PbDesc), ctypes.POINTER(_lib.DbpBand),
                                              ctypes.POINTER(cls), ctypes.POINTER(ctypes.c_void_p)]
    assert lib.pmx_pb_xpm_symbols.argtypes == [ctypes.c_void_p, ctypes.c_int32, ctypes.POINTER(ctypes.c_double)]
    assert {'pmx_pb_xpm_create', 'pmx_pb_xpm_symbols'} <= set(_lib.EXPORTS)


def test_python_arguments_are_checked():
    """ValueError for every refusal, the library's message where it is the library's, before any table is computed"""
    make_tx(256, 16, nch=3)
    fib = base_fiber()
    s = fiber_setup(fib, 'g-s-')
    with pytest.raises(ValueError, match='needs ich and decim'):
        pmx.pbnlc(fib, 'g-s-', 2, xpm='adjacent')
    with pytest.raises(ValueError, match='needs decim'):
        pbm.pb_plan(None, s, 2, xpm=[5])
    with pytest.raises(ValueError, match='xpm_coefs needs xpm'):
        pbm.pb_plan(None, s, 2, shift=0, decim=4, xpm_coefs=[([0], [0], [1.0])])
    for xpm, what in (([2], 'compensated channel itself'), ([4], 'does not exist'), ([1, 1], 'twice'), ('near', 'adjacent'),
                      ([], 'no interferer')):
        with pytest.raises(ValueError, match=what):
            pmx.pbnlc(fib, 'g-s-', 2, ich=2, decim=4, xpm=xpm)
    with pytest.raises(ValueError, match="pmx_pb_xpm_create: interferer 0 has the channel's own shift"):
        pbm.pb_plan(None, s, 2, shift=channel_ndfn(2), decim=4, xpm=[channel_ndfn(2)])
    with pytest.raises(ValueError, match='nint=9'):
        pbm.pb_plan(None, s, 2, shift=0, decim=4, xpm=list(range(1, 10)))
    with pytest.raises(ValueError, match=r'\|n\| at most 1024'):
        pbm.pb_plan(None, s, 2, shift=0, decim=4, xpm=[9], coefs=([0], [0], [1.0]), xpm_coefs=[([0], [2000], [1.0])])
    assert pbm.xpm_channels('adjacent', 1, 3) == [2] and pbm.xpm_channels('all', 2, 3) == [1, 3]


# ---------------------------------------------------------------------------------------------------------------- GPU
def _batch(gs, batch):
    """batch different realizations of the multiplex: shifted in time, the x polarization turned -> (x, y) [batch][1][nfft]"""
    xs = np.stack([np.roll(gs.FIELDX[:, 0], 7 * b) * np.exp(0.3j * b) for b in range(batch)])[:, None]
    ys = np.stack([np.roll(gs.FIELDY[:, 0], -5 * b) for b in range(batch)])[:, None]
    return np.ascontiguousarray(xs), np.ascontiguousarray(ys)


def _tables(s, nt, r, m, ints, K, nspan=2, prune=1e-6):
    """the channel's table and the XPM tables of its interferers (nquad 4: the stage is checked, not the physics)"""
    p = pbm.channel_pulse(nt, r, s.nfft)
    tab = pbm.pb_coefficients(pbm.channel_setup(s, m, r), nspan, p, K, prune, nt=nt // r, nquad=4)
    xt = [pbm.xpm_coefficients(s, nspan, m, c, r, p, K, nt=nt, nquad=4, prune=prune) for c in ints]
    return p, tab, xt


XPM = [  # nsymb, nt, decim, nch, ich, interferers, batch, manakov, K, prune
    (512, 16, 4, 3, 1, [2], 4, False, 16, 1e-6),              # 2^13 -> 2^11, edge of 3, one interferer
    (4096, 16, 16, 3, 2, [1, 3], 1, True, 0, 1e-6),           # 2^16 -> 2^12, centre of 3
    (2048, 32, 16, 9, 5, [1, 2, 3, 4, 6, 7, 8, 9], 1, False, 16, 1e-6),   # 2^16 -> 2^12, centre of 9 with all 8
    (65536, 16, 16, 3, 2, [3, 1], 16, True, 16, 1e-2),        # 2^20 -> 2^16, batch 16, interferers out of order (the
]                                                             # tables pruned: the numpy oracle is the cost here)


@pytest.mark.gpu
@pytest.mark.parametrize('case', XPM, ids=lambda c: '2^%d-r%d-nch%d-ch%d-int%d-b%d-%s-K%d' % (
    int(math.log2(c[0] * c[1])), c[2], c[3], c[4], len(c[5]), c[6], 'man' if c[7] else 'cnlse', c[8]))
def test_xpm_stage_matches_the_oracle(ctx, case):
    """A and every B (<= 1e-12), Delta against the oracle's triplets on the device's symbols (<= 1e-12) and the corrected
    field (<= 1e-10) against pb_xpm_channel, every realization its own field"""
    nsymb, nt, r, nch, ich, ints, batch, manakov, K, prune = case
    gs = make_tx(nsymb, nt, nch=nch, ftype='unique', pavg_mw=4.0)
    s = fiber_setup(base_fiber(slope=0.057), 'g-s-')
    s.manakov = manakov
    m, shifts = channel_ndfn(ich), [channel_ndfn(c) for c in ints]
    p, tab, xt = _tables(s, nt, r, m, shifts, K, prune=prune)
    w, gam = pbm.model_weights(s)
    wx, _ = pbm.xpm_weights(s)
    scale = pbm.scale_factor(s, 2, GAIN_DB)
    plan = pbm.pb_plan(ctx, s, 2, GAIN_DB, xi=0.8, K=K, batch=batch, nt=nt, coefs=tab, shift=m, decim=r, xpm=shifts,
                       xpm_coefs=xt)
    xs, ys = _batch(gs, batch)
    fld = _lib.DeviceField(ctx, s.nfft, 1, batch)
    fld.upload(xs, ys)
    plan.execute(fld)
    A, D = plan.symbols()
    Bs = [plan.xpm_symbols(c) for c in range(len(ints))]
    ox, oy = fld.download()
    plan.close()
    fld.close()
    a_ref, b_ref, u_dev, u_ref = [], [], [], []
    bins = dbp_oracle.channel_bins(s.nfft, m, r)
    for b in range(batch):
        rx, ry, ab, bb, _ = pxo.pb_xpm_channel(xs[b, 0], ys[b, 0], p, nt // r, tab, w, wx, gam, scale, 0.8, m, r,
                                               list(zip(shifts, xt)))
        a_ref.append(ab)
        b_ref.append(bb)
        bx, by = dbp_oracle.band_pass(xs[b, 0], bins), dbp_oracle.band_pass(ys[b, 0], bins)
        u_dev.append(np.concatenate([ox[b, 0] - bx, oy[b, 0] - by]))
        u_ref.append(np.concatenate([rx - bx, ry - by]))
    a_ref = np.stack(a_ref)
    d_dev = po.triplets(A, *tab, w, gam, scale)
    for B, t in zip(Bs, xt):
        d_dev = pxo.xpm_triplets(A, B, *t, wx, gam, scale, d_dev)
    eA = _rel(A, a_ref)
    eB = max(_rel(Bs[c], np.stack([bb[c] for bb in b_ref])) for c in range(len(ints)))
    eD, eU = _rel(D, d_dev), _rel(np.array(u_dev), np.array(u_ref))
    xpm_share = _rel(d_dev, po.triplets(A, *tab, w, gam, scale))
    print('pb xpm %s: ncoef %d + %s  A %.2e  B %.2e  Delta %.2e  correction %.2e  (|XPM| / |SPM| %.2f)'
          % (case, len(tab[2]), [len(t[2]) for t in xt], eA, eB, eD, eU, xpm_share))
    assert eA <= 1e-12 and eB <= 1e-12 and eD <= 1e-12 and eU <= 1e-10
    assert xpm_share > 1e-3


@pytest.mark.gpu
def test_xpm_stage_is_deterministic_xi0_is_the_band_pass_and_zero_tables_are_single_channel(ctx):
    """two executions give the same bits; xi = 0 is the band-pass and launches what single-channel PB-NLC at xi = 0
    launches (no interferer is extracted); tables of zeros give single-channel PB-NLC's bits"""
    nsymb, nt, r, batch, ich = 4096, 16, 8, 4, 2
    gs = make_tx(nsymb, nt, nch=3, ftype='unique', pavg_mw=4.0)
    s = fiber_setup(base_fiber(), 'g-s-')
    m, shifts = channel_ndfn(ich), [channel_ndfn(1), channel_ndfn(3)]
    p, tab, xt = _tables(s, nt, r, m, shifts, 16)
    zeros = [(t[0], t[1], np.zeros_like(t[2])) for t in xt]
    xs, ys = _batch(gs, batch)
    fld = _lib.DeviceField(ctx, s.nfft, 1, batch)
    runs = [('xpm', 1.0, xt), ('xpm', 1.0, xt), ('xpm', 0.0, xt), ('single', 0.0, None), ('xpm', 1.0, zeros),
            ('single', 1.0, None)]
    outs, launches = [], []
    for what, xi, t in runs:
        kw = dict(xpm=shifts, xpm_coefs=t) if what == 'xpm' else {}
        plan = pbm.pb_plan(ctx, s, 2, GAIN_DB, xi=xi, K=16, batch=batch, nt=nt, coefs=tab, shift=m, decim=r, **kw)
        fld.upload(xs, ys)
        n0 = ctx.launches
        plan.execute(fld)
        launches.append(ctx.launches - n0)
        plan.close()
        outs.append(fld.download())
    fld.close()
    same = lambda a, b: all(np.array_equal(a[i].view(np.uint64), b[i].view(np.uint64)) for i in range(2))
    print('launches (xpm, xpm, xpm xi=0, single xi=0, xpm zero tables, single):', launches)
    assert same(outs[0], outs[1])
    assert launches[2] == launches[3]
    bins = dbp_oracle.channel_bins(s.nfft, m, r)
    err = max(_rel(np.concatenate([outs[2][0][b, 0], outs[2][1][b, 0]]),
                   np.concatenate([dbp_oracle.band_pass(xs[b, 0], bins), dbp_oracle.band_pass(ys[b, 0], bins)]))
              for b in range(batch))
    assert err <= 1e-13
    assert same(outs[4], outs[5])
    assert not same(outs[0], outs[5])


def _multiplex(nsymb, nt, powers):
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
def test_xpm_pbnlc_lowers_the_residual_below_single_channel_pbnlc():
    """three channels at 1 mW each, 5 x 80 km, noise-free, decim 16: the centre channel's symbol-centre residual against its
    Tx (band-passed like the field) with XPM-aware PB-NLC is below single-channel PB-NLC's at the same K; CD, single-
    channel DBP and full-field DBP (one step per span) beside them.  (At 4 mW each CD alone leaves 1.8: the first-order
    model no longer holds there, and the larger XPM correction overshoots.)"""
    nsymb, nt, nspan, r, ich, K = 512, 32, 5, 16, 2, 32
    gs, _, _ = _multiplex(nsymb, nt, [1.0, 1.0, 1.0])
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
    for what in ('cd', 'pbnlc', 'pbnlc_xpm', 'dbp_channel', 'dbp_full'):
        G.FIELDX, G.FIELDY = ux.copy(), uy.copy()
        if what == 'cd':
            pmx.pbnlc(fib, 'g-s-', nspan, gain_db, xi=0.0, K=0, ich=ich, decim=r)
        elif what == 'pbnlc':
            pmx.pbnlc(fib, 'g-s-', nspan, gain_db, xi=1.0, K=K, ich=ich, decim=r)
        elif what == 'pbnlc_xpm':
            pmx.pbnlc(fib, 'g-s-', nspan, gain_db, xi=1.0, K=K, ich=ich, decim=r, xpm='adjacent', prune=1e-4)
        elif what == 'dbp_channel':
            pmx.dbp(fib, 'g-s-', nspan, gain_db, steps_per_span=1, ich=ich, decim=r)
        else:
            pmx.dbp(fib, 'g-s-', nspan, gain_db, steps_per_span=1)
            G.FIELDX = dbp_oracle.band_pass(np.asarray(G.FIELDX), bins)
            G.FIELDY = dbp_oracle.band_pass(np.asarray(G.FIELDY), bins)
        ox, oy = np.asarray(G.FIELDX)[::nt, 0], np.asarray(G.FIELDY)[::nt, 0]
        res[what] = math.sqrt((np.sum(np.abs(ox - tx) ** 2) + np.sum(np.abs(oy - ty) ** 2))
                              / (np.sum(np.abs(tx) ** 2) + np.sum(np.abs(ty) ** 2)))
    print('centre channel of three at 1 mW each, symbol-centre residual vs Tx: %s'
          % ', '.join('%s %.4f' % kv for kv in res.items()))
    assert res['pbnlc_xpm'] < res['pbnlc'] < res['cd']


COHMIX = {'oftype': 'gauss', 'obw': 1.9, 'eftype': 'bessel5', 'ebw': 0.65, 'lopower': 0.0}


@pytest.mark.gpu
def test_mc_cohmix_xpm_pbnlc_counts_fewer_errors(ctx):
    """the centre channel of three at 1 mW each, 20 x 80 km, amplifiers of 10 dB noise figure: McRunner('cohmix') with
    single-channel PB-NLC and xpm='adjacent' counts fewer errors than without, on the same realizations (at 6 mW each
    over 10 spans the first-order correction overshoots and counts more)"""
    nsymb, nt, nspan, nreal, batch, ich, r = 1 << 12, 16, 20, 16, 8, 2, 8
    _, sx, sy = _multiplex(nsymb, nt, [1.0, 1.0, 1.0])
    fib = dict(synth.SMF)
    fib.update(length=8e4, dgd=0.1, nplates=20, manakov='yes')
    setup = fiber_setup(fib, 'gps-', rng=np.random.Generator(np.random.PCG64(0)))
    G = pmx.GSTATE
    sym = np.stack([sx[:, ich - 1], sy[:, ich - 1]]).astype(np.uint8)
    out = {}
    for what, pb in (('spm', dict(K=32, decim=r)), ('xpm', dict(K=32, decim=r, xpm='adjacent', prune=1e-4))):
        run = mc.McRunner(ctx, setup, G.FIELDX_TX, G.FIELDY_TX, sym, nsymb, nt, nspan, GAIN_DB, 10.0, nreal, batch,
                          receiver='cohmix', dsp_params=dict(mu=1 / 2000, freqavg=200), rx_params=COHMIX, ich=ich,
                          compensation='pbnlc', pb_params=pb)
        try:
            out[what] = run.run(ase_seed=3)[0]
        finally:
            run.close()
    print('mc cohmix centre of three at equal powers: errors single-channel pbnlc %d, xpm-aware %d'
          % (out['spm'].sum(), out['xpm'].sum()))
    assert out['spm'].sum() > 0
    assert out['xpm'].sum() < out['spm'].sum()
