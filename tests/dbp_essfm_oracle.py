"""Enhanced split-step digital backpropagation restated in numpy (TEST INFRASTRUCTURE): the oracle of pmx_dbp_set_taps.

The existing DBP oracles (tests/dbp_oracle.py, dbp_pmd_oracle.py, dbp_scalar_oracle.py, dbp_channel_oracle.py) with one
change in every backward nonlinear step: each quantity it computes from |u|^2 is replaced by the circular FIR of real
taps c[0..2K] (c[K] at lag 0) in the time domain,
    q~[n] = sum_{m=-K..K} c[m+K] * q[(n - m) mod N]      (left to right in m),
as polmux_ssfm.h states it.  Two polarizations: the phase from the FIR of |ux|^2+|uy|^2, the CNLSE s3 rotation from the
FIR of s3, both taken from the field entering the step; scalar path: every |u_j|^2 of nl_step, with 'x' the sum over the
filtered powers.  The same step as tests/dbp_filtered_oracle.py with H = fft(c placed circularly), computed without a
transform.  taps = None runs the existing oracles themselves.  FP64; never imported by the product package.
"""
import numpy as np

import oracle.fiber_oracle as orc
import dbp_channel_oracle
import dbp_oracle
import dbp_pmd_oracle
import dbp_scalar_oracle


def fir(q, taps):
    """the circular FIR of every column of q, summed left to right in the lag m = -K..K (np.roll(q, m)[n] = q[n - m])"""
    c = np.asarray(taps, dtype=np.float64).ravel()
    k = c.size // 2
    out = np.zeros_like(q)
    for j in range(c.size):
        out = out + c[j] * np.roll(q, j - k, axis=0)
    return out


def circular_response(nfft, taps):
    """fft of the taps placed circularly on a grid of nfft samples (c[K] at 0, c[K+m] at m mod nfft): the H with which
    filtered DBP computes the same step"""
    c = np.asarray(taps, dtype=np.float64).ravel()
    k = c.size // 2
    h = np.zeros(nfft)
    for j in range(c.size):
        h[(j - k) % nfft] += c[j]
    return np.fft.fft(h)


def matrix_nl_step_fir(ismanakov, alphalin, gam, dz, ux, uy, nfc, taps):
    """orc.matrix_nl_step (spm) with the FIR of the power and s3"""
    leff = orc._leff(alphalin, dz, np.float64)
    p = ux.real ** 2 + ux.imag ** 2 + uy.real ** 2 + uy.imag ** 2
    s3 = 2 * (ux.real * uy.imag - ux.imag * uy.real)
    pf = fir(p, taps)
    s3f = None if ismanakov else fir(s3, taps)
    for k in range(nfc):
        gamleff = np.float64(gam[k]) * leff
        e = orc.fastexp(-gamleff * pf[:, k])
        ux[:, k] = ux[:, k] * e
        uy[:, k] = uy[:, k] * e
        if not ismanakov:
            e = orc.fastexp(gamleff * s3f[:, k] / 3)
            c, s = e.real, e.imag
            ux[:, k], uy[:, k] = c * ux[:, k] + s * uy[:, k], -s * ux[:, k] + c * uy[:, k]
    return ux, uy


def nl_step_fir(alphalin, gam, dz, u, nfc, spm, xpm, taps):
    """orc.nl_step with the FIR of every |u_j|^2"""
    leff = orc._leff(alphalin, dz, np.float64)
    powr = fir(u.real ** 2 + u.imag ** 2, taps)
    if xpm:
        tot = np.sum(powr, axis=1, keepdims=True) * np.ones((1, nfc))
        powr = 2 * tot - powr if spm else 2 * (tot - powr)
    elif not spm:
        return u
    return u * orc.fastexp(-gam * powr * leff)


def _gain(u, gain):
    return u if gain is None else u * (1.0 / np.sqrt(gain))


def dbp(ux, uy, betat, gam, alphalin, nfc, lf, manakov, spm=1, nspan=1, gain=None, steps_per_span=None, step_len=None,
        span_steps=None, xi=1.0, taps=None):
    """dbp_oracle.dbp with the FIR in the nonlinear step"""
    if taps is None:
        return dbp_oracle.dbp(ux, uy, betat, gam, alphalin, nfc, lf, manakov, spm, nspan, gain, steps_per_span, step_len,
                              span_steps, xi)
    ux = np.array(ux, dtype=np.complex128, copy=True)
    uy = np.array(uy, dtype=np.complex128, copy=True)
    g = -float(xi) * np.asarray(gam, dtype=np.float64)
    if manakov == 'yes':
        g = g * 8 / 9
    betat = np.asarray(betat, dtype=np.float64).reshape(ux.shape[0], nfc)
    spans = dbp_pmd_oracle._spans(nspan, lf, steps_per_span, step_len, span_steps)
    for k in reversed(range(nspan)):
        ux, uy = _gain(ux, gain), _gain(uy, gain)
        for h in reversed(spans[k]):
            a = np.exp(0.5 * alphalin * h)
            ux = orc.lin_step(-betat * h, ux * a)
            uy = orc.lin_step(-betat * h, uy * a)
            if spm:
                ux, uy = matrix_nl_step_fir(manakov == 'yes', alphalin, g, h, ux, uy, nfc, taps)
    return ux, uy


def dbp_pmd(ux, uy, betat, db1, gam, alphalin, nfc, lf, manakov, brfs, spm=1, nspan=1, gain=None, steps_per_span=None,
            step_len=None, span_steps=None, xi=1.0, taps=None):
    """dbp_pmd_oracle.dbp_pmd with the FIR in the nonlinear step"""
    if taps is None:
        return dbp_pmd_oracle.dbp_pmd(ux, uy, betat, db1, gam, alphalin, nfc, lf, manakov, brfs, spm, nspan, gain,
                                      steps_per_span, step_len, span_steps, xi)
    ux = np.array(ux, dtype=np.complex128, copy=True)
    uy = np.array(uy, dtype=np.complex128, copy=True)
    g = -float(xi) * np.asarray(gam, dtype=np.float64)
    if manakov == 'yes':
        g = g * 8 / 9
    nplates = len(brfs[0]['theta'])
    lcorr = lf / nplates
    nbt = -np.asarray(betat, dtype=np.float64).reshape(ux.shape[0], nfc)
    ndb1 = -np.asarray(db1, dtype=np.float64).reshape(ux.shape[0], nfc)
    spans = dbp_pmd_oracle._spans(nspan, lf, steps_per_span, step_len, span_steps)
    for k in reversed(range(nspan)):
        ux, uy = _gain(ux, gain), _gain(uy, gain)
        rb = dbp_pmd_oracle.reversed_brf(brfs[k])
        part = dbp_pmd_oracle.forward_partition(spans[k], lf, nplates)
        for h, st in zip(reversed(spans[k]), reversed(part)):
            a = np.exp(0.5 * alphalin * h)
            ux, uy = ux * a, uy * a
            ntr = st['ntrunk']
            first = nplates - (st['ntot'] - st['nmem']) - ntr
            if ntr > 0:
                ux, uy = orc.matrix_step(nbt, ndb1, st['dzb'][::-1], ntr, ux, uy, rb, first, 0, lcorr, np.float64)
            if spm:
                ux, uy = matrix_nl_step_fir(manakov == 'yes', alphalin, g, h, ux, uy, nfc, taps)
    return ux, uy


def dbp_scalar(u, betat, gam, alphalin, nfc, lf, spm=1, xpm=0, nspan=1, gain=None, steps_per_span=None, step_len=None,
               span_steps=None, xi=1.0, taps=None):
    """dbp_scalar_oracle.dbp_scalar with the FIR in the nonlinear step"""
    if taps is None:
        return dbp_scalar_oracle.dbp_scalar(u, betat, gam, alphalin, nfc, lf, spm, xpm, nspan, gain, steps_per_span,
                                            step_len, span_steps, xi)
    u = np.array(u, dtype=np.complex128, copy=True)
    nfft = u.shape[0]
    g = (-float(xi) * np.asarray(gam, dtype=np.float64)).reshape(1, -1) * np.ones((nfft, 1))
    betat = np.asarray(betat, dtype=np.float64).reshape(nfft, nfc)
    spans = dbp_scalar_oracle._spans(nspan, lf, steps_per_span, step_len, span_steps)
    for k in reversed(range(nspan)):
        u = _gain(u, gain)
        for h in reversed(spans[k]):
            u = orc.lin_step(-betat * h, u * np.exp(0.5 * alphalin * h))
            u = nl_step_fir(alphalin, g, h, u, nfc, spm, xpm, taps)
    return u


def dbp_channel(ux, uy, betat, gam, alphalin, lf, manakov, shift, decim, db1=None, brfs=None, spm=1, taps=None, **kw):
    """dbp_channel_oracle.dbp_channel with the FIR on the channel's M-sample grid (a tap spans decim samples of the
    full field)"""
    if taps is None:
        return dbp_channel_oracle.dbp_channel(ux, uy, betat, gam, alphalin, lf, manakov, shift, decim, db1, brfs, spm, **kw)
    C = dbp_channel_oracle
    nfft = ux.shape[0]
    b = C.channel_bins(nfft, shift, decim)
    cx, cy = C.crop(ux, b, decim), C.crop(uy, b, decim)
    bt = np.asarray(betat, dtype=np.float64).reshape(nfft, 1)[b]
    if brfs is None:
        vx, vy = dbp(cx, cy, bt, gam, alphalin, 1, lf, manakov, spm=spm, taps=taps, **kw)
    else:
        d1 = np.asarray(db1, dtype=np.float64).reshape(nfft, 1)[b]
        vx, vy = dbp_pmd(cx, cy, bt, d1, gam, alphalin, 1, lf, manakov, brfs, spm=spm, taps=taps, **kw)
    return C.embed(vx, b, nfft, decim), C.embed(vy, b, nfft, decim)
