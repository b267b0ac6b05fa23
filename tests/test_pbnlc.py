"""Perturbation-based nonlinearity compensation (polmux_b200/pbnlc.py, pmx_pb_create / pmx_pb_exec, tests/pbnlc_oracle.py).

On the CPU: the table is the link's first-order term (against the forward oracle), the FFT form of the table against the
direct overlap integral, the ABI mirror and the validation.  On the GPU: the device stage against the oracle on both
resident layouts, determinism, xi = 0, and the compensation a receive chain gets from it."""
import ctypes
import importlib
import math
import os
import subprocess

import numpy as np
import pytest

import oracle.fiber_oracle as orc
import pbnlc_oracle as po
import polmux_b200 as pmx
from polmux_b200 import _lib, mc, synth
from polmux_b200.fiber import fiber_setup
from common import base_fiber, make_tx

pbm = importlib.import_module('polmux_b200.pbnlc')
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _link(nsymb, nt, pavg_mw, nspan, manakov, length=8e4):
    """noise-free oracle link of nspan spans, the gain exp(alpha*L) after each -> (Tx (x, y), CD-compensated Rx (x, y), setup)"""
    gs = make_tx(nsymb, nt, pavg_mw=pavg_mw)
    s = fiber_setup(base_fiber(length=length, dphimax=1e-3), 'g-s-')
    s.manakov = manakov
    g = math.exp(s.alphalin * s.length)
    ux, uy = gs.FIELDX.copy(), gs.FIELDY.copy()
    for _ in range(nspan):
        _, _, ux, uy, _, _ = orc.matrix_ssfm(ux, uy, s.betat, s.db1, s.dzmaxt, s.dphimaxt, s.gam, s.alphalin, 1, s.length, 1,
                                             'yes' if manakov else 'no', s.fls, s.brf)
        ux, uy = ux * math.sqrt(g), uy * math.sqrt(g)
    bt = s.betat * (s.length * nspan)
    return (gs.FIELDX, gs.FIELDY), (orc.lin_step(-bt, ux), orc.lin_step(-bt, uy)), s


def _mismatch(pavg_mw, manakov, K=32, nsymb=256, nt=8, nspan=3):
    """|Delta_meas - Delta_pred| / |Delta_meas| of the projected symbols"""
    tx, rx, s = _link(nsymb, nt, pavg_mw, nspan, manakov)
    p = synth.cosroll_pulse(nt, 0.2)
    a_tx, a_rx = po.project(*tx, p, nt), po.project(*rx, p, nt)
    m, n, C = pbm.pb_coefficients(s, nspan, p, K, nt=nt)
    w, gam = pbm.model_weights(s)
    d_meas, d_pred = a_rx - a_tx, po.triplets(a_tx, m, n, C, w, gam)
    return np.linalg.norm(d_meas - d_pred) / np.linalg.norm(d_meas)


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize('manakov', [False, True])
def test_table_is_the_links_first_order_term(manakov):
    """3 x 80 km, no noise, dphimax 1e-3, K = 32: the projected perturbation of the forward oracle against the triplet sum of
    the table on the Tx symbols.  Measured: 0.131 / 0.068 / 0.062 (CNLSE) at 2 / 0.5 / 0.125 mW.  The floor of about 6 %
    is the part of the first-order term the triplet form leaves out (the products whose indices do not satisfy
    i + j - l = k, which an NRZ pulse of one symbol's width does not make negligible); above it the mismatch is second
    order: once the floor is taken out (in quadrature) it shrinks about 4x when the power is divided by 4."""
    e = [_mismatch(p, manakov) for p in (2.0, 0.5, 0.125)]
    print('first-order mismatch (manakov=%s) at 2 / 0.5 / 0.125 mW: %s' % (manakov, ['%.4f' % v for v in e]))
    assert e[2] < 0.08
    hi, lo = math.sqrt(e[0] ** 2 - e[2] ** 2), math.sqrt(max(e[1] ** 2 - e[2] ** 2, 0.0))
    assert 3.0 < hi / lo < 5.5, (e, hi / lo)


def test_fast_table_equals_the_direct_overlap_integral():
    """the FFT form of pb_coefficients against the term-by-term integral of the oracle, both on the whole block"""
    make_tx(128, 8)
    s = fiber_setup(base_fiber(length=4e4, slope=0.057), 'g-s-')
    p = synth.cosroll_pulse(8, 0.2)
    K = 3
    m, n, C = pbm.pb_coefficients(s, 2, p, K, nt=8, nquad=8, window=128)
    Cd = po.coefficients_direct(s.betat[:, 0], s.length, s.alphalin, 2, p, 8, K, 8)
    Cf = C.reshape(2 * K + 1, 2 * K + 1)
    assert np.array_equal(m.reshape(Cf.shape)[:, 0], np.arange(-K, K + 1))
    assert np.abs(Cf - Cd).max() <= 1e-12 * abs(Cd[K, K])
    assert np.array_equal(Cf, Cf.T)
    assert np.abs(Cd - Cd.T).max() <= 1e-12 * abs(Cd[K, K])


def test_table_converges_with_the_quadrature_and_prunes():
    """the table against 64 nodes per span falls with every doubling of the nodes (measured 1.2e-2, 4.5e-3, 1.6e-3 of the
    largest entry at 8, 16, 32: algebraic, the overlaps of the sharp-edged pulse are not smooth in z at the start of the
    link); pruning keeps the large entries and the symmetry"""
    make_tx(256, 8)
    s = fiber_setup(base_fiber(), 'g-s-')
    p = synth.cosroll_pulse(8, 0.2)
    C = {q: pbm.pb_coefficients(s, 3, p, 8, nt=8, nquad=q)[2] for q in (8, 16, 32, 64)}
    d = [np.abs(C[q] - C[64]).max() / abs(C[64]).max() for q in (8, 16, 32)]
    print('quadrature: max |C(q) - C(64)| / max |C| for q = 8, 16, 32:', d)
    assert d[0] > 2 * d[1] > 4 * d[2] and d[2] < 3e-3
    m, n, Cp = pbm.pb_coefficients(s, 3, p, 8, prune=1e-2, nt=8)
    c00 = abs(C[32][C[32].size // 2])
    assert 0 < Cp.size < C[32].size and np.abs(Cp).min() >= 1e-2 * c00
    assert np.array_equal(np.sort(m * 100 + n), np.sort(n * 100 + m))      # the pruned table stays symmetric


def test_default_window_matches_the_whole_block():
    """the table on the default window equals the table on the whole block"""
    make_tx(1024, 8)
    s = fiber_setup(base_fiber(), 'g-s-')
    p = synth.cosroll_pulse(8, 0.2)
    w = pbm.default_window(s, 2, p, 8, 8)
    assert w < 1024
    a = pbm.pb_coefficients(s, 2, p, 8, nt=8, nquad=8)[2]
    b = pbm.pb_coefficients(s, 2, p, 8, nt=8, nquad=8, window=1024)[2]
    assert np.abs(a - b).max() <= 1e-6 * np.abs(b).max()


def test_oracle_stage_identities():
    """xi = 0 returns the field; a field built from symbol amplitudes on orthogonal pulses projects back onto them"""
    rng = np.random.default_rng(3)
    N, nt = 256, 8
    ux, uy = rng.standard_normal((2, N)) + 1j * rng.standard_normal((2, N))
    p = synth.cosroll_pulse(nt, 0.2)
    rx, ry, _, _ = po.stage(ux, uy, p, nt, [0], [0], [1.0 + 0.5j], pbm.CNLSE, 1e-3, 1.0, 0.0)
    assert np.array_equal(rx, ux) and np.array_equal(ry, uy)
    box = np.r_[np.zeros(nt // 2), np.ones(nt), np.zeros(nt // 2)]      # non-overlapping pulses
    a = rng.standard_normal((2, N // nt)) + 0j
    vx, vy = po.reconstruct(np.zeros(N), np.zeros(N), -a, box, nt, 1.0)
    assert np.abs(po.project(vx, vy, box, nt) - a).max() < 1e-14


def test_pb_structs_match_the_header(tmp_path):
    """gcc probe against the header: pmx_pb_desc equals its ctypes mirror"""
    cls = _lib.PbDesc
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "polmux_ssfm.h"', 'int main(void){',
             'printf("size %zu\\n", sizeof(pmx_pb_desc));']
    for fname, _ in cls._fields_:
        lines.append('printf("%s %%zu\\n", offsetof(pmx_pb_desc, %s));' % (fname, fname))
    lines += ['printf("maxk %d\\n", PMX_PB_MAX_K);', 'return 0;}']
    src = tmp_path / 'probe.c'
    src.write_text('\n'.join(lines))
    exe = tmp_path / 'probe'
    subprocess.run(['gcc', '-I', os.path.join(ROOT, 'include'), str(src), '-o', str(exe)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(out['size']) == ctypes.sizeof(cls)
    for fname, _ in cls._fields_:
        assert int(out[fname]) == getattr(cls, fname).offset, fname
    assert int(out['maxk']) == _lib.PB_MAX_K


def _desc(**kw):
    nsymb, nt = kw.pop('nsymb', 64), kw.pop('nt', 16)
    m, n, C = kw.pop('m', [0, 1]), kw.pop('n', [0, -1]), kw.pop('C', [1.0, 0.5j])
    d, keep = _lib.make_pb(nsymb, nt, 1, synth.cosroll_pulse(nt, 0.2), pbm.CNLSE, 1.3e-3, 1.0, 1.0, m, n, C)
    for k, v in kw.items():
        setattr(d, k, v)
    return d, keep


def test_pb_create_rejects_bad_descriptors_without_a_context():
    lib = _lib.load()
    bad = {
        'nfc=2': (dict(nfc=2), _lib.PMX_ERR_UNSUPPORTED),
        'FP64 fields only': (dict(precision=_lib.PMX_F32), _lib.PMX_ERR_UNSUPPORTED),
        'must equal nfft': (dict(nfft=2048), _lib.PMX_ERR_INVALID),
        'at most 128': (dict(m=[129], n=[0], C=[1.0]), _lib.PMX_ERR_INVALID),
        'coefficient 1 is not finite': (dict(C=[1.0, complex(float('nan'), 0)]), _lib.PMX_ERR_INVALID),
        'batch must be': (dict(batch=0), _lib.PMX_ERR_INVALID),
        'npulse=3': (dict(npulse=3), _lib.PMX_ERR_INVALID),
        'ncoef=0': (dict(ncoef=0), _lib.PMX_ERR_INVALID),
        'must be finite': (dict(xi=float('inf')), _lib.PMX_ERR_INVALID),
    }
    for what, (kw, code) in bad.items():
        d, keep = _desc(**kw)
        h = ctypes.c_void_p()
        rc = lib.pmx_pb_create(None, ctypes.byref(d), ctypes.byref(h))
        msg = lib.pmx_last_error(None).decode()
        assert rc == code and what in msg, (what, rc, msg)
        assert not h.value


def test_pbnlc_and_mcrunner_refuse_what_they_cannot_run():
    make_tx(256, 16, nch=3, ftype='unique')
    with pytest.raises(ValueError, match='one channel'):
        pmx.pbnlc(base_fiber(), 'g-s-', 2)
    make_tx(256, 16)
    with pytest.raises(ValueError, match='at most 128'):
        pmx.pbnlc(base_fiber(), 'g-s-', 2, K=200)
    with pytest.raises(ValueError, match='wrong flag'):
        pmx.pbnlc(base_fiber(), 'g-s', 2)
    s = fiber_setup(base_fiber(), 'g-s-')
    with pytest.raises(ValueError, match="compensation='pbnlc' needs"):
        mc.McRunner(None, s, None, None, np.zeros((2, 256), np.uint8), 256, 16, 1, 16.0, 5.0, 2, 2, receiver='genie',
                    compensation='pbnlc')
    with pytest.raises(ValueError, match="pb_params needs"):
        mc.McRunner(None, s, None, None, np.zeros((2, 256), np.uint8), 256, 16, 1, 16.0, 5.0, 2, 2, receiver='blind',
                    compensation='cd', pb_params=dict(xi=0.5))


# ---------------------------------------------------------------------------------------------------------------- GPU
def _fields(nfft, batch, seed):
    """batch different seeded PDM-QPSK fields at a few mW -> (x, y) [batch][1][nfft]"""
    nt = 16 if nfft >= 1 << 10 else 8
    xs, ys = [], []
    for b in range(batch):
        ex, ey, _, _ = synth.pdm_qpsk(nfft // nt, nt, 1, seed_x=seed + 2 * b, seed_y=seed + 2 * b + 1)
        r = np.random.default_rng(seed + b)
        xs.append(2.0 * ex[:, 0] + 0.1 * (r.standard_normal(nfft) + 1j * r.standard_normal(nfft)))
        ys.append(2.0 * ey[:, 0] + 0.1 * (r.standard_normal(nfft) + 1j * r.standard_normal(nfft)))
    return np.array(xs)[:, None], np.array(ys)[:, None]


def _table(nsymb, nt, K, prune, manakov):
    make_tx(nsymb, nt)
    s = fiber_setup(base_fiber(), 'g-s-')
    s.manakov = manakov
    return s, pbm.pb_coefficients(s, 2, synth.cosroll_pulse(nt, 0.2), K, prune, nt=nt, nquad=8)


def _rel(a, b):
    return float(np.linalg.norm(np.ravel(a) - np.ravel(b)) / np.linalg.norm(np.ravel(b)))


STAGE = [  # nfft, nt, batch, manakov, K, prune
    (1 << 10, 16, 1, False, 0, 0.0),
    (1 << 10, 16, 16, True, 4, 0.0),
    (1 << 10, 8, 1, False, 64, 0.0),
    (1 << 10, 16, 16, False, 32, 1e-3),
    (1 << 16, 16, 1, True, 64, 1e-3),
    (1 << 16, 16, 16, False, 4, 0.0),
    (1 << 16, 16, 1, False, 32, 0.0),
    (1 << 16, 16, 16, True, 64, 1e-2),
    (1 << 20, 16, 1, False, 16, 1e-3),
]


@pytest.mark.gpu
@pytest.mark.parametrize('nfft,nt,batch,manakov,K,prune', STAGE)
def test_device_stage_matches_the_oracle(ctx, nfft, nt, batch, manakov, K, prune):
    """projection, triplet sum (<= 1e-12) and the corrected field (<= 1e-10) against the oracle, every realization its own
    field; both resident layouts (natural below 2^12 samples, transposed from 2^12)"""
    nsymb = nfft // nt
    s, (m, n, C) = _table(nsymb, nt, K, prune, manakov)
    w, gam = pbm.model_weights(s)
    p = synth.cosroll_pulse(nt, 0.2)
    scale, xi = 1.7, 0.8
    xs, ys = _fields(nfft, batch, 11)
    fld = _lib.DeviceField(ctx, nfft, 1, batch)
    fld.upload(xs, ys)
    plan = _lib.PbPlan(ctx, _lib.make_pb(nsymb, nt, batch, p, w, gam, xi, scale, m, n, C))
    plan.execute(fld)
    A, D = plan.symbols()
    ox, oy = fld.download()
    plan.close()
    fld.close()
    a_ref = np.stack([po.project(xs[b, 0], ys[b, 0], p, nt) for b in range(batch)])
    d_ref = po.triplets(A, m, n, C, w, gam, scale)
    eA, eD = _rel(A, a_ref), _rel(D, d_ref)
    cx, cy = [], []
    for b in range(batch):
        rx, ry = po.reconstruct(xs[b, 0], ys[b, 0], D[b], p, nt, xi)
        cx.append(rx - xs[b, 0])
        cy.append(ry - ys[b, 0])
    eU = _rel(np.concatenate([ox[:, 0] - xs[:, 0], oy[:, 0] - ys[:, 0]]), np.concatenate([np.array(cx), np.array(cy)]))
    full = po.triplets(a_ref, m, n, C, w, gam, scale)                  # the whole chain from the oracle's own projection
    eF = _rel(D, full)
    print('pb stage nfft=%d batch=%d K=%d ncoef=%d: A %.2e  Delta %.2e  Delta(oracle A) %.2e  correction %.2e'
          % (nfft, batch, K, len(C), eA, eD, eF, eU))
    assert eA <= 1e-12 and eD <= 1e-12 and eF <= 1e-10 and eU <= 1e-10


@pytest.mark.gpu
def test_device_stage_is_deterministic_and_xi0_is_a_no_op(ctx):
    nfft, nt, batch = 1 << 16, 16, 4
    s, (m, n, C) = _table(nfft // nt, nt, 32, 0.0, False)
    w, gam = pbm.model_weights(s)
    p = synth.cosroll_pulse(nt, 0.2)
    xs, ys = _fields(nfft, batch, 5)
    fld = _lib.DeviceField(ctx, nfft, 1, batch)
    outs = []
    for xi in (1.0, 1.0, 0.0):
        fld.upload(xs, ys)
        plan = _lib.PbPlan(ctx, _lib.make_pb(nfft // nt, nt, batch, p, w, gam, xi, 1.0, m, n, C))
        plan.execute(fld)
        plan.close()
        outs.append(fld.download())
    fld.upload(xs, ys)
    ref = fld.download()                                                  # the upload / download round trip
    fld.close()
    assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1])
    assert not np.array_equal(outs[0][0], ref[0])
    assert np.array_equal(outs[2][0].view(np.uint64), ref[0].view(np.uint64))
    assert np.array_equal(outs[2][1].view(np.uint64), ref[1].view(np.uint64))


@pytest.mark.gpu
def test_device_stage_refuses_a_field_it_was_not_made_for(ctx):
    d, keep = _desc(nsymb=64, nt=16)
    plan = _lib.PbPlan(ctx, (d, keep))
    for kw, what in ((dict(nfft=2048, nfc=1, batch=1), 'nfft=2048'), (dict(nfft=1024, nfc=1, batch=2), 'batch 2'),
                     (dict(nfft=1024, nfc=2, batch=1), 'nfc=2')):
        fld = _lib.DeviceField(ctx, **kw)
        with pytest.raises(_lib.PolmuxError, match=what):
            plan.execute(fld)
        fld.close()
    plan.close()


def _symbol_residual(G, tx, s_scale, nt):
    ux, uy = np.asarray(G.FIELDX)[::nt, 0] * s_scale, np.asarray(G.FIELDY)[::nt, 0] * s_scale
    return math.sqrt((np.sum(np.abs(ux - tx[0][::nt, 0]) ** 2) + np.sum(np.abs(uy - tx[1][::nt, 0]) ** 2))
                     / (np.sum(np.abs(tx[0][::nt, 0]) ** 2) + np.sum(np.abs(tx[1][::nt, 0]) ** 2)))


@pytest.mark.gpu
@pytest.mark.parametrize('manakov', [False, True])
def test_pbnlc_lowers_the_residual_below_cd_only(ctx, manakov):
    """one channel, 5 x 80 km at 4 mW, where the nonlinear distortion dominates, noise-free: the symbol-centre residual against Tx after pmx.pbnlc is below that of the all-pass step alone; DBP at one
    step per span beside it"""
    nsymb, nt, nspan = 1024, 8, 5
    tx, rx, s = _link(nsymb, nt, 4.0, nspan, manakov)
    gain_db = 10 * math.log10(math.exp(s.alphalin * s.length))
    fib = base_fiber(dphimax=1e-3)
    flag = 'gps-' if manakov else 'g-s-'          # (pbnlc and dbp drop the 'p': Manakov with x.manakov = 'yes', no plates)
    if manakov:
        fib.update(manakov='yes', dgd=0.0)
    G = pmx.GSTATE
    res = {}
    for what in ('cd', 'pbnlc', 'dbp'):
        bt = s.betat * (s.length * nspan)
        G.FIELDX, G.FIELDY = orc.lin_step(bt, rx[0]), orc.lin_step(bt, rx[1])    # the received field, dispersed again
        if what == 'cd':
            pmx.pbnlc(fib, flag, nspan, gain_db, xi=0.0, K=0)
        elif what == 'pbnlc':
            pmx.pbnlc(fib, flag, nspan, gain_db, xi=1.0, K=48)
        else:
            pmx.dbp(fib, flag, nspan, gain_db, steps_per_span=1)
        res[what] = _symbol_residual(G, tx, 1.0, nt)
    print('symbol-centre residual vs Tx (manakov=%s): CD only %.4f, PB-NLC (K=48) %.4f, DBP 1 step/span %.4f'
          % (manakov, res['cd'], res['pbnlc'], res['dbp']))
    assert res['pbnlc'] < 0.8 * res['cd']


def _mc_scenario(nsymb, nt, pavg_mw):
    ex, ey, sx, sy = synth.pdm_qpsk(nsymb, nt, 1)
    pmx.reset_all(nsymb, nt, 1)
    G = pmx.GSTATE
    G.SYMBOLRATE, G.LAMBDA, G.POWER = 28.0, np.array([1550.0]), np.array([float(pavg_mw)])
    pmx.create_field('unique', ex, ey, {'power': 'average'})
    fib = dict(synth.SMF)
    fib.update(length=8e4, dgd=0.1, nplates=20, manakov='yes')
    setup = fiber_setup(fib, 'gps-', rng=np.random.Generator(np.random.PCG64(0)))
    return G, setup, np.stack([sx[:, 0], sy[:, 0]]).astype(np.uint8)


@pytest.mark.gpu
def test_mcrunner_with_pbnlc(ctx):
    """McRunner(compensation='pbnlc'): with xi = 0 the counts and CMA pass counts of compensation='cd'; with xi = 1 fewer
    errors than 'cd' on the same realizations at a launch power where the nonlinear distortion dominates (10 x 80 km at
    12 mW; measured on a B200: 38768 errors with 'cd', 34074 with 'pbnlc', 58532 with DBP at one step per span)"""
    nsymb, nt, nspan, nreal, batch = 1 << 12, 16, 10, 16, 8
    G, setup, sym = _mc_scenario(nsymb, nt, 12.0)
    dspp = dict(mu=1 / 2000, freqavg=200)
    out = {}
    for what, comp, pb in (('cd', 'cd', None), ('xi0', 'pbnlc', dict(xi=0.0, K=8)), ('pb', 'pbnlc', dict(xi=1.0, K=48)),
                           ('dbp', 'dbp', None)):
        r = mc.McRunner(ctx, setup, G.FIELDX_TX, G.FIELDY_TX, sym, nsymb, nt, nspan, 16.0, 5.0, nreal, batch,
                        receiver='blind', dsp_params=dspp, compensation=comp, pb_params=pb)
        counts, _ = r.run(ase_seed=3)
        out[what] = (counts, list(r.passes))
        r.close()
    print('mc errors: cd %d, pbnlc %d, dbp (1 step/span) %d' % (out['cd'][0].sum(), out['pb'][0].sum(), out['dbp'][0].sum()))
    assert np.array_equal(out['xi0'][0], out['cd'][0])
    assert [np.asarray(p).tolist() for p in out['xi0'][1]] == [np.asarray(p).tolist() for p in out['cd'][1]]
    assert out['cd'][0].sum() > 0
    assert out['pb'][0].sum() < out['cd'][0].sum()
