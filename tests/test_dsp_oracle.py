"""The DSP oracle (oracle/dsp_oracle.py) pinned against the reference's own M source, executed by the mini interpreter:
cmaadaptivefilter.m, samp2pat.m, pat_decoder.m (+ pat2stars.m, stars2pat.m, fastshift.m, nmod.m) and the sub-functions
vitvit / cmapolardemux of dsp4cohdec.m.  CPU only; the pins need the toolbox's M source and skip without it."""
import os

import numpy as np
import pytest

import oracle.dsp_oracle as dsp
from oracle.mini_m.interp import Interp, MStruct, to_m

REF = '/root/reference'
needs_ref = pytest.mark.skipif(not os.path.exists(os.path.join(REF, 'dsp4cohdec.m')), reason='reference tree not present')


def _signals(L, seed, rot=0.3, noise=0.05, dphi=2e-3):
    """two mixed, noisy, slowly rotating QPSK streams (one sample per symbol)"""
    g = np.random.Generator(np.random.PCG64(seed))
    sym = (g.integers(0, 2, (L, 2)) * 2 - 1 + 1j * (g.integers(0, 2, (L, 2)) * 2 - 1)) / np.sqrt(2)
    mix = np.array([[np.cos(rot), np.sin(rot) * np.exp(0.4j)], [-np.sin(rot) * np.exp(-0.4j), np.cos(rot)]])
    x = sym @ mix.T + noise * (g.standard_normal((L, 2)) + 1j * g.standard_normal((L, 2)))
    return x * np.exp(1j * (0.2 + dphi * np.arange(L)))[:, None], sym


@needs_ref
def test_cmaadaptivefilter_matches_reference_source():
    x, _ = _signals(200, 1)
    ext = np.concatenate([x[-3:], x, x[:3]])
    h1 = np.zeros((7, 2), dtype=complex)
    h2 = np.zeros((7, 2), dtype=complex)
    h1[3, 0] = 1
    h2[3, 1] = 1
    it = Interp(REF)
    y, a, b = it.call('cmaadaptivefilter', [ext, h1, h2, to_m(7), to_m(1 / 600), np.array([[1.0, 1.0]]), to_m(1)], 3)
    yo, ao, bo = dsp.cma_adaptive_filter(ext, h1, h2, 1 / 600, (1.0, 1.0))
    np.testing.assert_allclose(yo, y, rtol=0, atol=1e-14)
    np.testing.assert_allclose(ao, a, rtol=0, atol=1e-14)
    np.testing.assert_allclose(bo, b, rtol=0, atol=1e-14)


def _local(it, name, args, nargout=1):
    table = it.load('dsp4cohdec')
    return it.call(name, args, nargout, local_funcs=table)


@needs_ref
@pytest.mark.parametrize('P,M,k,unwrap', [(4, 4, 20, False), (2, 4, 3, True), (4, 4, 0, True), (2, 4, 300, True)])
def test_vitvit_matches_reference_source(P, M, k, unwrap):
    x, _ = _signals(256, 2)
    it = Interp(REF)
    ref = _local(it, 'vitvit', [x, to_m(P), to_m(M), to_m(k), to_m(bool(unwrap))])[0]
    got = dsp.vitvit(x, P, M, k, unwrap)
    np.testing.assert_allclose(got, ref, rtol=0, atol=2e-12)


@needs_ref
def test_cmapolardemux_matches_reference_source():
    x, _ = _signals(300, 3, rot=0.25)
    it = Interp(REF)
    params = MStruct({'R': np.array([[1.0, 1.0]]), 'mu': to_m(1 / 300), 'taps': to_m(5), 'txpolars': to_m(2), 'phizero': to_m(0.0)})
    ref = _local(it, 'cmapolardemux', [x, params])[0]
    got, passes = dsp.cma_polar_demux(x, mu=1 / 300, taps=5, R=(1.0, 1.0), phizero=0.0)
    assert passes >= 2
    np.testing.assert_allclose(got, ref, rtol=0, atol=1e-11)


@needs_ref
def test_easiadaptivefilter_matches_reference_source():
    x, _ = _signals(200, 5, rot=0.5)
    h1 = np.array([[1.0, 0.2j]])
    h2 = np.array([[-0.2j, 1.0]])
    it = Interp(REF)
    y, a, b = it.call('easiadaptivefilter', [x, h1, h2, to_m(1), to_m(1 / 300), to_m(1)], 3)
    yo, ao, bo = dsp.easi_adaptive_filter(x, h1, h2, 1 / 300)
    np.testing.assert_allclose(yo, y, rtol=0, atol=1e-13)
    np.testing.assert_allclose(ao, a, rtol=0, atol=1e-13)
    np.testing.assert_allclose(bo, b, rtol=0, atol=1e-13)


@needs_ref
def test_easipolardemux_matches_reference_source():
    x, _ = _signals(300, 6, rot=0.6)
    it = Interp(REF)
    params = MStruct({'mu': to_m(1 / 300), 'txpolars': to_m(2), 'phizero': to_m(0.1)})
    ref = _local(it, 'easipolardemux', [x, params])[0]
    got, passes = dsp.easi_polar_demux(x, mu=1 / 300, phizero=0.1)
    assert passes >= 2
    np.testing.assert_allclose(got, ref, rtol=0, atol=1e-11)


@needs_ref
def test_dispcompfilter_matches_reference_source():
    it = Interp(REF)
    beta2l = -800.0 * 1550.0 ** 2 / 2 / np.pi / 299792458.0 * 1e-21
    for n, flen in ((256, 16), (512, 32)):
        ref = np.asarray(_local(it, 'DispCompFilter', [to_m(beta2l), to_m(28e9), to_m(n), to_m(flen)])[0]).ravel()
        got = dsp.disp_comp_filter(beta2l, 28e9, n, flen)
        np.testing.assert_allclose(got, ref, rtol=0, atol=1e-12)
        assert abs(np.abs(got).mean() - 1) < 0.2          # close to an all-pass response


@needs_ref
def test_nlrotation_matches_reference_source():
    x, _ = _signals(128, 7)
    x = x * (1 + 0.3 * np.random.Generator(np.random.PCG64(8)).standard_normal((128, 1)))
    it = Interp(REF)
    ref = _local(it, 'NLRotation', [x, to_m(0.37)])[0]
    np.testing.assert_allclose(dsp.nl_rotation(x, 0.37), ref, rtol=0, atol=1e-14)


@needs_ref
def test_adc_emulation_matches_reference_source():
    """the ADC lines of dsp4cohdec.m sit in its main body: they are cut out of the file as text and executed"""
    import re
    from oracle.mini_m.interp import Parser, tokenize
    src = open(os.path.join(REF, 'dsp4cohdec.m'), encoding='latin-1').read()
    m = re.search(r"if p\.applyadc(.*?)\nend", src, re.S)
    assert m and 'round' in m.group(1)
    fn = 'function Irx = adcwrap(Irx, p)\n' + m.group(1) + '\n'
    f = Parser(tokenize(fn), 'adcwrap.m').parse_file()[0]
    it = Interp(REF)
    irx = np.random.Generator(np.random.PCG64(9)).standard_normal((200, 4)) * 3.0
    for bits in (3, 5, 8):
        ref = it.run_function(f, [irx, MStruct({'adcbits': to_m(bits)})], 1, {'adcwrap': f})[0]
        got = dsp.adc_quantize(irx, bits)
        np.testing.assert_allclose(got, ref, rtol=0, atol=1e-15)
        assert len(np.unique(np.round(got, 12))) <= 2 ** bits + 1


@needs_ref
def test_decision_and_differential_decoding_match_reference_source():
    g = np.random.Generator(np.random.PCG64(4))
    phase = g.uniform(-np.pi, np.pi, (64, 2))
    it = Interp(REF)
    x = MStruct({'rec': 'coherent'})
    s = MStruct({'logic': np.array([[0.0], [1.0]]), 'thr': to_m(0.0)})
    ref = it.call('samp2pat', [x, s, phase], 1)[0]
    got = dsp.samp2pat_coherent(phase)
    np.testing.assert_array_equal(got, np.asarray(ref).astype(np.uint8))
    for cols in ((0, 2), (2, 4)):
        pm = got[:, cols[0]:cols[1]].astype(np.float64)
        rp, rpm = it.call('pat_decoder', [pm, 'dqpsk', MStruct({'binary': to_m(True)})], 2)
        op, opm = dsp.pat_decoder_dqpsk_binary(pm)
        np.testing.assert_array_equal(op, np.asarray(rp).ravel().astype(np.int64))
        np.testing.assert_array_equal(opm, np.asarray(rpm).astype(np.int64))


def test_blind_chain_recovers_the_symbols():
    """CMA + carrier recovery + differential decision on a mixed, rotating, noisy stream: no errors"""
    x, sym = _signals(2048, 5, rot=0.35, noise=0.03, dphi=1e-3)
    y, passes = dsp.cma_polar_demux(x, mu=1 / 2000, taps=7)
    ph = dsp.carrier_recovery(y, 2, 100, 3, 2)
    assert dsp.count_errors_dqpsk(ph, np.angle(sym)) == 0
    # and errors are counted when the noise is large
    x2, sym2 = _signals(2048, 6, rot=0.35, noise=0.35, dphi=1e-3)
    y2, _ = dsp.cma_polar_demux(x2, mu=1 / 2000, taps=7)
    assert dsp.count_errors_dqpsk(dsp.carrier_recovery(y2, 2, 100, 3, 2), np.angle(sym2)) > 0
