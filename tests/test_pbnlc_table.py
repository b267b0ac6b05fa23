"""The PB-NLC triplet table on the device (pmx_pb_table; pbnlc.pb_coefficients(ctx=), pb_plan / pmx.pbnlc(table='device')).

On the CPU: the ctypes mirror against the header, and every refusal of a bad descriptor without a context.  On the GPU:
the device table against the numpy table of pb_coefficients on both resident layouts, single-channel included; its window,
symmetry and determinism; and the stage and the Monte-Carlo receiver with either table."""
import ctypes
import importlib
import math
import os
import subprocess

import numpy as np
import pytest

import polmux_b200 as pmx
from polmux_b200 import _lib, mc, synth
from polmux_b200.fiber import fiber_setup
from polmux_b200.receiver import channel_ndfn
from common import base_fiber, make_tx, rel_l2

pbm = importlib.import_module('polmux_b200.pbnlc')
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _desc(**kw):
    """a valid descriptor (2^10 samples, nt 16, 2 spans, K 4), with the fields in kw overridden"""
    nfft, nt = 1024, 16
    d, keep = _lib.make_pb_table(nfft, nt, np.linspace(-1e-3, 1e-3, nfft), synth.cosroll_pulse(nt, 0.2), 2, 8e4, 4.6e-5,
                                 4, 8, 0, 0.0)
    for k, v in kw.items():
        if k == 'betat_values':
            keep['betat_bad'] = np.ascontiguousarray(v, dtype=np.float64)
            d.betat = keep['betat_bad'].ctypes.data_as(ctypes.POINTER(ctypes.c_double))
        elif k == 'pulse_values':
            keep['pulse_bad'] = np.ascontiguousarray(v, dtype=np.float64)
            d.pulse = keep['pulse_bad'].ctypes.data_as(ctypes.POINTER(ctypes.c_double))
            d.npulse = keep['pulse_bad'].size
        else:
            setattr(d, k, v)
    return d, keep


def _table_rc(d, null=None):
    """pmx_pb_table without a context -> (code, message); null names one output passed as NULL"""
    lib = _lib.load()
    cap = (2 * max(int(d.K), 0) + 1) ** 2
    m, n = np.zeros(cap, np.int32), np.zeros(cap, np.int32)
    coef = np.zeros(2 * cap)
    cnt = ctypes.c_int32(0)
    ip = ctypes.POINTER(ctypes.c_int32)
    args = {'m': m.ctypes.data_as(ip), 'n': n.ctypes.data_as(ip),
            'coef': coef.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), 'ncoef': ctypes.byref(cnt)}
    if null:
        args[null] = None
    rc = lib.pmx_pb_table(None, ctypes.byref(d), args['m'], args['n'], args['coef'], args['ncoef'], None)
    return rc, lib.pmx_last_error(None).decode()


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_table_desc_and_prototype_match_the_header(tmp_path):
    """a gcc probe against the header: pmx_pb_table_desc's size and offsets equal the ctypes mirror, and the prototype
    compiles with the argument types the binding passes"""
    cls = _lib.PbTableDesc
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "polmux_ssfm.h"',
             'static int (*fn)(pmx_ctx*, const pmx_pb_table_desc*, int32_t*, int32_t*, double*, int32_t*, int32_t*) = '
             'pmx_pb_table;', 'int main(void){', 'printf("size %zu\\n", sizeof(pmx_pb_table_desc));']
    for fname, _ in cls._fields_:
        lines.append('printf("%s %%zu\\n", offsetof(pmx_pb_table_desc, %s));' % (fname, fname))
    lines.append('return fn == 0;}')
    src = tmp_path / 'probe.c'
    src.write_text('\n'.join(lines))
    exe = tmp_path / 'probe'
    subprocess.run(['gcc', '-Werror', '-I', os.path.join(ROOT, 'include'), str(src), '-o', str(exe),
                    '-Wl,--unresolved-symbols=ignore-all'], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True).stdout.splitlines())
    assert int(out['size']) == ctypes.sizeof(cls)
    for fname, _ in cls._fields_:
        assert int(out[fname]) == getattr(cls, fname).offset, fname
    assert 'pmx_pb_table' in _lib.EXPORTS and hasattr(_lib.load(), 'pmx_pb_table')


def test_table_rejects_bad_descriptors_without_a_context():
    """every refusal comes without a context, with its code and message; a valid request gets as far as the missing
    context"""
    nan = float('nan')
    cases = [  # descriptor fields, code, message
        (dict(K=-1), _lib.PMX_ERR_INVALID, 'K=-1, |m| and |n| at most 128'),
        (dict(K=129), _lib.PMX_ERR_INVALID, 'K=129'),
        (dict(nquad=0), _lib.PMX_ERR_INVALID, 'nquad=0'),
        (dict(nspan=0), _lib.PMX_ERR_INVALID, 'nspan=0'),
        (dict(nspan=1 << 16, nquad=32), _lib.PMX_ERR_INVALID, 'nodes, at most 2^20'),
        (dict(length=0.0), _lib.PMX_ERR_INVALID, 'span length must be finite and positive'),
        (dict(length=-8e4), _lib.PMX_ERR_INVALID, 'span length must be finite and positive'),
        (dict(length=math.inf), _lib.PMX_ERR_INVALID, 'span length must be finite and positive'),
        (dict(alphalin=-1e-5), _lib.PMX_ERR_INVALID, 'alphalin must be finite and non-negative'),
        (dict(alphalin=nan), _lib.PMX_ERR_INVALID, 'alphalin must be finite and non-negative'),
        (dict(prune=nan), _lib.PMX_ERR_INVALID, 'prune must be finite'),
        (dict(prune=math.inf), _lib.PMX_ERR_INVALID, 'prune must be finite'),
        (dict(betat_values=np.r_[np.zeros(1023), nan]), _lib.PMX_ERR_INVALID, 'betat[1023] is not finite'),
        (dict(betat=None), _lib.PMX_ERR_INVALID, 'null betat'),
        (dict(window=3), _lib.PMX_ERR_INVALID, 'the window (3 symbols) must divide the block (64 symbols)'),
        (dict(window=-2), _lib.PMX_ERR_INVALID, 'the window (-2 symbols) must divide'),
        (dict(window=2), _lib.PMX_ERR_UNSUPPORTED, 'a window of 32 samples, at least 2^6'),
        (dict(nt=3), _lib.PMX_ERR_INVALID, 'nt=3 must divide nfft'),
        (dict(nt=0), _lib.PMX_ERR_INVALID, 'nt=0 must divide nfft'),
        (dict(nfft=1000), _lib.PMX_ERR_INVALID, 'nfft=1000, built for powers of two'),
        (dict(nfft=32), _lib.PMX_ERR_INVALID, 'nfft=32, built for powers of two'),
        (dict(pulse_values=np.ones(3)), _lib.PMX_ERR_INVALID, 'npulse=3'),
        (dict(pulse_values=np.ones(512)), _lib.PMX_ERR_INVALID, 'npulse=512'),
        (dict(pulse_values=np.r_[1.0, nan]), _lib.PMX_ERR_INVALID, 'pulse sample 1 is not finite'),
        (dict(pulse_values=np.zeros(4)), _lib.PMX_ERR_INVALID, 'the pulse has no energy'),
        (dict(pulse=None), _lib.PMX_ERR_INVALID, 'npulse='),
    ]
    for fields, code, msg in cases:
        rc, err = _table_rc(_desc(**fields)[0])
        assert rc == code and msg in err, (fields, rc, err)
    for null in ('m', 'n', 'coef', 'ncoef'):
        rc, err = _table_rc(_desc()[0], null=null)
        assert rc == _lib.PMX_ERR_INVALID and 'pmx_pb_table: null argument' in err, null
    rc, err = _table_rc(_desc()[0])
    assert rc == _lib.PMX_ERR_INVALID and 'null ctx' in err
    rc, err = _table_rc(_desc(window=8, K=128)[0])          # a window smaller than the lags is the host's too
    assert rc == _lib.PMX_ERR_INVALID and 'null ctx' in err


def test_python_table_argument_is_checked():
    make_tx(64, 16)
    s = fiber_setup(base_fiber(), 'g-s-')
    with pytest.raises(ValueError, match="table must be 'host'"):
        pbm.pb_plan(None, s, 2, table='gpu')
    with pytest.raises(ValueError, match="table must be 'host'"):
        pmx.pbnlc(base_fiber(), 'g-s-', 2, table='numpy')
    with pytest.raises(ValueError, match='K=200'):               # pb_table checks through the library without a device
        pbm.pb_table(None, s, 2, synth.cosroll_pulse(16, 0.2), K=200)
    with pytest.raises(ValueError, match='must divide the block'):    # the same exception type as the host path
        pbm.pb_table(None, s, 2, synth.cosroll_pulse(16, 0.2), K=4, window=3)
    with pytest.raises(ValueError, match='must divide the block'):
        pbm.pb_coefficients(s, 2, None, 4, nt=16, window=3)


# ---------------------------------------------------------------------------------------------------------------- GPU
TABLE_CASES = [  # nsymb, nt, nspan, K, nquad, window, prune
    (64, 16, 1, 0, 8, None, 0.0),                  # 2^10, natural layout
    (64, 16, 10, 4, 32, None, 0.0),
    (64, 16, 3, 4, 8, 16, 0.0),                    # explicit window
    (1024, 16, 3, 16, 32, None, 0.0),              # 2^14, transposed
    (1024, 16, 1, 32, 8, 512, 0.0),
    (2048, 8, 3, 16, 8, None, 1e-3),               # pruned
    (256, 64, 3, 16, 8, None, 0.0),                # more phases than one step holds
    (4096, 16, 1, 32, 8, 512, 0.0),                # 2^16
    (4096, 16, 10, 4, 8, None, 0.1),
]


def _case_setup(nsymb, nt):
    make_tx(nsymb, nt)
    return fiber_setup(base_fiber(slope=0.057), 'g-s-')


def _compare(dev, host, label):
    (m, n, C), (mh, nh, Ch) = dev, host
    assert np.array_equal(m, mh) and np.array_equal(n, nh), label
    c00 = abs(Ch[(mh == 0) & (nh == 0)][0])
    err = np.abs(C - Ch).max() / c00
    print('%s: %d entries, max |dC| / |C00| = %.2e' % (label, C.size, err))
    assert err <= 1e-12, (label, err)


@pytest.mark.gpu
@pytest.mark.parametrize('case', TABLE_CASES, ids=lambda c: 'n%dx%d_s%d_K%d_q%d_w%s_p%g' % c)
def test_device_table_matches_the_host_table(ctx, case):
    nsymb, nt, nspan, K, nquad, window, prune = case
    s = _case_setup(nsymb, nt)
    p = synth.cosroll_pulse(nt, 0.2)
    host = pbm.pb_coefficients(s, nspan, p, K, prune, nt, nquad, window)
    if prune:   # no entry so close to the threshold that rounding could move it across
        full = pbm.pb_coefficients(s, nspan, p, K, 0.0, nt, nquad, window)[2]
        r = np.abs(full) / abs(full[full.size // 2])
        assert np.abs(r - prune).min() > 1e-9 * prune
        assert 0 < host[2].size < full.size
    m, n, C, W = pbm.pb_table(ctx, s, nspan, p, K, prune, nt, nquad, window)
    assert W == (window or pbm.default_window(s, nspan, p, nt, K))
    _compare((m, n, C), host, 'table %s' % (case,))
    if not prune:
        T = C.reshape(2 * K + 1, 2 * K + 1)
        assert np.array_equal(T, T.T)
    assert all(np.array_equal(a, b) for a, b in zip(pbm.pb_table(ctx, s, nspan, p, K, prune, nt, nquad, window),
                                                     (m, n, C, W)))        # two calls, the same bits


@pytest.mark.gpu
def test_device_table_of_a_single_channel(ctx):
    """the table of channel_setup with the pulse of channel_pulse, for an edge channel of three at decim 8"""
    make_tx(1024, 16, nch=3, ftype='unique')
    s = fiber_setup(base_fiber(slope=0.057), 'g-s-')
    r = 8
    cs, p = pbm.channel_setup(s, channel_ndfn(3, pmx.GSTATE), r), pbm.channel_pulse(16, r, s.nfft)
    host = pbm.pb_coefficients(cs, 3, p, 8, nt=16 // r, nquad=8)
    dev = pbm.pb_coefficients(cs, 3, p, 8, nt=16 // r, nquad=8, ctx=ctx)
    _compare(dev, host, 'single-channel table')


@pytest.mark.gpu
@pytest.mark.parametrize('nsymb', [64, 1024])
def test_stage_with_the_device_table_matches_the_host_table(ctx, nsymb):
    """pmx.pbnlc(table='device') against table='host' on the same received field: the same correction to rounding"""
    nt, nspan = 16, 3
    make_tx(nsymb, nt, pavg_mw=4.0)
    G = pmx.GSTATE
    fib = base_fiber()
    x0, y0 = G.FIELDX.copy(), G.FIELDY.copy()
    out = {}
    for table in ('host', 'device'):
        G.FIELDX, G.FIELDY = x0.copy(), y0.copy()
        pmx.pbnlc(fib, 'g-s-', nspan, 16.0, K=16, table=table)
        out[table] = (np.asarray(G.FIELDX).copy(), np.asarray(G.FIELDY).copy())
    err = rel_l2(*out['device'], *out['host'])
    corr = rel_l2(*out['host'], x0, y0)
    print('stage device vs host table: rel_l2 %.2e (the correction itself %.2e)' % (err, corr))
    assert corr > 1e-6 and err <= 1e-12


@pytest.mark.gpu
def test_mcrunner_counts_the_same_errors_with_either_table(ctx):
    """McRunner('cohmix', compensation='pbnlc', pb_params with table) on the centre channel of three, 10 x 80 km at 12 mW
    between neighbours at 2 mW: the same error counts with the host and the device table"""
    tpc = importlib.import_module('test_pbnlc_channel')
    nsymb, nt, nspan, nreal, batch, ich, r = 1 << 12, 16, 10, 4, 2, 2, 8
    fib, setup, sx, sy = tpc._mc_link(nsymb, nt, [2.0, 12.0, 2.0], 0.1)
    G = pmx.GSTATE
    sym = np.stack([sx[:, ich - 1], sy[:, ich - 1]]).astype(np.uint8)
    out = {}
    for table in ('host', 'device'):
        run = mc.McRunner(ctx, setup, G.FIELDX_TX, G.FIELDY_TX, sym, nsymb, nt, nspan, tpc.GAIN_DB, 5.0, nreal, batch,
                          receiver='cohmix', dsp_params=dict(mu=1 / 2000, freqavg=200), rx_params=tpc.COHMIX, ich=ich,
                          compensation='pbnlc', pb_params=dict(K=16, decim=r, table=table))
        try:
            out[table] = run.run(ase_seed=3)[0]
        finally:
            run.close()
    print('mc cohmix errors with the host / device table: %d / %d' % (out['host'].sum(), out['device'].sum()))
    assert out['host'].sum() > 0 and np.array_equal(out['host'], out['device'])
