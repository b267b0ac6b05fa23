"""Front-end of the coherent receiver on the device: receiver_cohmix(ich, x) -- receiver_cohmix.m:1.

    post fiber + OBPF  ->  90-degree hybrids with the local oscillator  ->  photodiodes  ->  LPF

The parameter arithmetic stays on the host as in the reference (channel position, the post-fiber's betat, the two
filter responses from myfilter over GSTATE.FN, the LO vector); everything per sample runs on the GPU on a copy of the
channel's field column: the shift of the channel to baseband (pmx_field_modulate), the two filters (filter plans,
pmx_filter_create: the same three passes as a linear fiber step), the four mixer outputs and the photocurrents
(pmx_cohmix_exec).  GSTATE is left unchanged (receiver_cohmix.m:60-61)."""
from __future__ import annotations

import math

import numpy as np

from . import _lib
from . import gstate
from .gstate import CONSTANTS, GSTATE

_R4P2R2 = 2.61312592975275
_B1, _B2, _B3 = 3.86370330515627315, 7.4641016151377546, 9.1416201726856413
_BB = 0.3863
_D0, _D1, _D2, _D3, _D4 = 945.0, 945.0, 420.0, 105.0, 15.0


def myfilter(ftype, f, bw, ord_=0):
    """Hf = myfilter(ftype, f, bw, ord): myfilter.m:73-152, a column over the frequencies f (normalised like bw)."""
    x = np.asarray(f, dtype=np.float64).ravel() / bw
    ftype = str(ftype).lower()
    if ftype == 'movavg':
        return np.sinc(x).astype(np.complex128)
    if ftype == 'gauss':
        return np.exp(-0.5 * math.log(2) * x * x).astype(np.complex128)
    if ftype == 'gauss_off':
        return np.exp(-0.5 * math.log(2) * (x - ord_ / bw) * (x - ord_ / bw)).astype(np.complex128)
    if ftype == 'butt2':
        return 1.0 / (1 - x * x + 1j * math.sqrt(2) * x)
    if ftype == 'butt4':
        x2 = x * x
        umx2 = 1 - x2
        return 1.0 / (umx2 * umx2 - math.sqrt(2) * x2 + 1j * _R4P2R2 * x * umx2)
    if ftype == 'butt6':
        x2 = x * x
        x3 = x2 * x
        x4 = x3 * x
        x5 = x4 * x
        x6 = x5 * x
        return 1.0 / (1.0 - _B2 * x2 + _B2 * x4 - x6 + 1j * (_B1 * x - _B3 * x3 + _B1 * x5))
    if ftype == 'ideal':
        return (np.abs(x) <= 1).astype(np.complex128)
    if ftype == 'bessel5':
        om = 2 * math.pi * x * _BB
        om2 = om * om
        om3 = om2 * om
        om4 = om3 * om
        om5 = om4 * om
        return _D0 / ((_D0 - _D2 * om2 + _D4 * om4) + 1j * (_D1 * om - _D3 * om3 + om5))
    if ftype == 'rc1':
        return 1.0 / (1 + 1j * x)
    if ftype == 'rc2':
        return 1.0 / (1 + 1j * math.sqrt(math.sqrt(2) - 1) * x) ** 2
    if ftype == 'supergauss':
        if not ord_:
            raise ValueError('missing superGauss order')
        return np.exp(-0.5 * math.log(2) * x ** (2 * ord_)).astype(np.complex128)
    raise ValueError('the filter ftype does not exist.')


def evaldelay(ftype, bw):
    """group delay of the filter at f = 0, in symbols: evaldelay.m:28-80"""
    ftype = str(ftype).lower()
    if ftype in ('movavg', 'gauss', 'gauss_off', 'ideal', 'supergauss'):
        return 0.0
    if ftype == 'butt2':
        return 1.11 * math.sqrt(2) / (2 * math.pi * bw)
    if ftype == 'butt4':
        return 1.1 * _R4P2R2 / (2 * math.pi * bw)
    if ftype == 'butt6':
        return 1.1 * _B1 / (2 * math.pi * bw)
    if ftype == 'bessel5':
        return _BB / bw
    if ftype == 'rc1':
        return 1 / (2 * math.pi * bw)
    if ftype == 'rc2':
        return (math.sqrt(2) - 1) / (math.pi * bw)
    raise ValueError('the filter ftype does not exist.')


def hermitian_part(h):
    """(H(f) + conj(H(-f)))/2 over an FFT-ordered grid: real(ifft(fft(I).*H)) of a REAL sequence I equals ifft(fft(I).*Hh),
    which lets two real currents ride one complex transform (receiver_cohmix.m:297-300)."""
    h = np.asarray(h, dtype=np.complex128).ravel()
    mirror = np.conj(np.roll(h[::-1], 1))
    return 0.5 * (h + mirror)


def channel_ndfn(ich, G=None):
    """The offset of channel ich in a field holding every channel (receiver_cohmix.m:85-105), in FFT bins: the shift
    pmx_field_modulate takes to bring the channel to baseband (its spectrum sits on the bins k - ndfn)."""
    G = G or GSTATE
    fn = np.asarray(G.FN, dtype=np.float64).ravel()
    lam = np.asarray(G.LAMBDA, dtype=np.float64).ravel()
    maxl, minl = lam.max(), lam.min()
    lamc = 2 * maxl * minl / (maxl + minl)
    minfreq = fn[1] - fn[0]
    return round(CONSTANTS.CLIGHT * (1 / lamc - 1 / lam[ich - 1]) / G.SYMBOLRATE / minfreq)


class CohmixSetup:
    """What receiver_cohmix.m:78-169,178-219 derives from (ich, x) and GSTATE before it touches the samples."""

    def __init__(self, ich, x, G=None, nfc=None, randn=None):
        G = G or GSTATE
        x = self.x = dict(x)
        x.setdefault('oord', 0)                                               # receiver_cohmix.m:69-75
        x.setdefault('eord', 0)
        clight = CONSTANTS.CLIGHT
        fn = np.asarray(G.FN, dtype=np.float64).ravel()
        nfft = self.nfft = fn.size
        nfc = G.field_shape()[1] if nfc is None else nfc
        lam = np.asarray(G.LAMBDA, dtype=np.float64).ravel()
        maxl, minl = lam.max(), lam.min()
        lamc = 2 * maxl * minl / (maxl + minl)
        if ich > G.NCH or ich < 1:
            raise ValueError('The channel does not exist')
        if nfc != G.NCH:                                                      # one field for all the channels (:85-105)
            self.ndfn = int(channel_ndfn(ich, G))
            self.nch = 1
            self.ndfnl = nfft // 2 if ich == 1 else int(round((self.ndfn - channel_ndfn(ich - 1, G)) * 0.5))
            self.ndfnr = nfft // 2 if ich == G.NCH else int(round((channel_ndfn(ich + 1, G) - self.ndfn) * 0.5))
        else:
            self.ndfn, self.nch, self.ndfnl, self.ndfnr = 0, ich, nfft // 2, nfft // 2
        self.b2b = False
        if 'b2b' in x:                                                        # :113-122
            if x['b2b'] != 'b2b':
                raise ValueError("the b2b field must be 'b2b'")
            self.b2b = True
            x.pop('dpost', None)
        if 'dpost' in x:                                                      # post-compensating fiber (:139-166)
            lm = x['lambda']
            b20z = -lm ** 2 / 2 / math.pi / clight * x['dpost'] * 1e-3
            b30z = (lm / 2 / math.pi / clight) ** 2 * (2 * lm * x['dpost'] + lm ** 2 * x['slopez']) * 1e-3
            d_i0 = 2 * math.pi * clight * (1.0 / lam[ich - 1] - 1 / lm)
            d_ic = 2 * math.pi * clight * (1.0 / lam[ich - 1] - 1 / lamc)
            d_c0 = 2 * math.pi * clight * (1.0 / lamc - 1 / lm)
            beta1z = b20z * d_ic + 0.5 * b30z * (d_i0 ** 2 - d_c0 ** 2)
            beta2z = b20z + b30z * d_i0
            omega = 2 * math.pi * G.SYMBOLRATE * fn
            betat = omega * beta1z + 0.5 * omega ** 2 * beta2z + omega ** 3 * b30z / 6
            x['post_delay'] = G.SYMBOLRATE * beta1z
            hf = np.cos(betat) - 1j * np.sin(betat)                           # fastexp(-betat)
        else:
            hf = np.ones(nfft, dtype=np.complex128)
            x['post_delay'] = 0
        self.hf_opt = hf * myfilter(x['oftype'], fn, 0.5 * x['obw'], x['oord'])          # :169
        self.hf_el = myfilter(x['eftype'], fn, x['ebw'], x['eord'])                      # :293
        # local oscillator (:178-219)
        self.detune = 0.0
        if x.get('lodetuning'):
            minfreq = G.SYMBOLRATE * 1e9 / G.NSYMB
            kdet = math.floor(x['lodetuning'] / minfreq)
            if not kdet:
                import warnings
                warnings.warn('Detuning is neglected! Minimum frequency too high.')
            self.detune = 2 * math.pi * kdet / nfft
        self.lophase = None
        if 'lophasenoise' in x:
            ph = np.asarray(x['lophasenoise'], dtype=np.float64).ravel()
            if ph.size != nfft:
                raise ValueError('Incompatible vector.')
            self.lophase = ph
        elif 'lolinewidth' in x:
            draw = randn if randn is not None else (lambda n: gstate.rng().standard_normal(n))
            fnz = np.ones(nfft) * math.sqrt(2 * math.pi * x['lolinewidth'] / G.NT) * draw(nfft)
            fnz[0] = 0
            ph = np.cumsum(fnz)
            # Brownian bridge (:212-214): the loop reads LO_PhaseNoise(end) anew in every turn, but only its last turn changes it
            self.lophase = ph - np.arange(nfft) / (nfft - 1) * ph[-1]
        self.ecw = 10 ** (x['lopower'] / 20) if 'lopower' in x else 1.0
        self.balanced = not (x.get('pdtype') == 'normal')                     # :264-268


def front_end(ich, x, ctx, want_energy=False, randn=None):
    """The device part of receiver_cohmix: -> (DeviceField [1][1][Nfft] whose X / Y slots hold I + i*Q of the two
    polarizations' currents, CohmixSetup, x updated).  The caller closes the field."""
    G = GSTATE
    nfr, nfc = G.field_shape()
    S = CohmixSetup(ich, x, G, nfc, randn)
    isy = G.has_y()
    xo = S.x
    col = _lib.DeviceField(ctx, S.nfft, 1, 1)
    try:
        if S.b2b:                                                            # the transmitted field (:124-128, 224-229)
            tx = np.asarray(G.FIELDX_TX)[:, S.nch - 1]
            ty = None
            if isy and G.FIELDY_TX is not None and np.size(G.FIELDY_TX):
                ty = np.asarray(G.FIELDY_TX)[:, S.nch - 1]
            col.upload(tx[:, None], None if ty is None else ty[:, None])
        elif isy:
            fld, hx, hy = G.take_device(ctx, _lib.PMX_F64)
            try:
                _lib.field_copy_cols(col, 0, fld, S.nch - 1, 1)
            finally:
                G.restore_host(fld, hx, hy)
        else:
            col.upload(np.asarray(G.FIELDX)[:, S.nch - 1:S.nch], None)
        if S.ndfn:
            _lib.field_modulate(ctx, col, S.ndfn)
        if want_energy:   # normalised average energy per bit in the channel's band, before the optical filter (:174-175,233-234)
            band = np.zeros(S.nfft)
            band[:S.ndfnl] = 1
            band[S.nfft - S.ndfnr:] = 1
            tmp = _lib.DeviceField(ctx, S.nfft, 1, 1)
            try:
                _lib.field_copy_cols(tmp, 0, col, 0, 1)
                if not band.all():       # energy of the channel's band only: Parseval on the band-limited copy
                    f_ = _lib.Filter(ctx, S.nfft, 1, band)
                    try:
                        f_.execute(tmp)
                    finally:
                        f_.close()
                px, py = _lib.field_mean_power_xy(ctx, tmp)
            finally:
                tmp.close()
            pch = float(np.asarray(G.POWER).ravel()[ich - 1])
            xo['avgebx'] = px[0, 0] / pch
            if isy:
                xo['avgeby'] = py[0, 0] / pch
        fo = _lib.Filter(ctx, S.nfft, 1, S.hf_opt)
        try:
            fo.execute(col)
        finally:
            fo.close()
        _lib.cohmix_exec(ctx, col, S.ecw, S.detune, S.lophase, S.balanced)
        fe = _lib.Filter(ctx, S.nfft, 1, hermitian_part(S.hf_el))
        try:
            fe.execute(col)
        finally:
            fe.close()
    except Exception:
        col.close()
        raise
    return col, S, xo


def receiver_cohmix(ich, x, ctx=None, nargout=1, randn=None):
    """Iric = receiver_cohmix(ich, x): the photocurrents of channel ich, [Nfft, 2] (X: in-phase, quadrature) or
    [Nfft, 4] (X, then Y) -- receiver_cohmix.m:1.  With nargout = 2 also returns x with avgebx / avgeby / post_delay."""
    ctx = ctx or _lib.default_context()
    isy = GSTATE.has_y()
    col, S, xo = front_end(ich, x, ctx, want_energy=nargout >= 2, randn=randn)
    try:
        zx, zy = col.download()
    finally:
        col.close()
    cur = [zx[0, 0].real, zx[0, 0].imag]
    if isy:
        cur += [zy[0, 0].real, zy[0, 0].imag]
    iric = np.ascontiguousarray(np.stack(cur, axis=1))
    return (iric, xo) if nargout >= 2 else iric
