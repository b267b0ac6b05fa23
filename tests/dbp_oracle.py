"""Digital backpropagation restated in numpy (TEST INFRASTRUCTURE): the oracle of pmx_dbp_create / pmx_dbp_exec,
pmx_dbp_channel_create, pmx_dbp_set_filter and pmx_dbp_set_taps.

The reference has no DBP, so there is no reference source to pin this against.  It is built from the pinned forward
oracle's own operators -- matrix_nl_step (fiber.m:827-874), nl_step (fiber.m:787-804), lin_step (fiber.m:771-773),
checkstep (fiber.m:739-758), matrix_step (fiber.m:904-935) and _leff -- in the order polmux_ssfm.h documents, and tied to
the forward oracle by the exact inverse: with the forward run's own steps, xi = 1 and no noise, it returns the transmitted
field up to rounding, PMD and XPM included (tests/test_dbp*.py).  PMD-aware DBP at xi = 0 with one step per span is also
the pinned inverse_pmd (inverse_pmd_chain).

The nonlinear-step intensity is a keyword of every entry point (at most one; none is plain DBP, the forward oracle's own
step): each quantity the step computes from |u|^2 -- the power and, CNLSE, s3 of the field entering the step; on the
scalar path every |u_j|^2, with 'x' the sum of the filtered powers -- is replaced by
- bw: filtered DBP, ifft(fft(q) .* H) with the Gaussian H[k] = exp(-(ln 2/2) (k_s/bw)^2) at the signed bin k_s;
- taps: enhanced split-step DBP, the circular FIR q~[n] = sum_{m=-K..K} c[m+K] q[(n - m) mod N] (left to right in m),
  computed without a transform; it equals filtered DBP with H = circular_response(N, taps);
- response: filtered DBP with an explicit per-bin H.
On a single channel it acts on the channel's M-sample grid (the same bw in bins; a tap spans decim samples of the full
field).  Written for a real dtype chosen by the caller (the single-channel oracles FP64 only); never imported by the
product package.
"""
import math

import numpy as np

import oracle.fiber_oracle as orc


# ------------------------------------------------------------------------------------------------------------ schedule
def _spans(nspan, lf, steps_per_span, step_len, span_steps):
    """every span's steps in forward order: steps_per_span uniform steps of lf/steps_per_span, or step_len -- one span's
    steps for every span, or with span_steps [nspan] all spans' steps concatenated"""
    if step_len is None:
        m = int(steps_per_span or 1)
        return [[lf / m] * m for _ in range(nspan)]
    if span_steps is None:
        return [list(np.asarray(step_len, dtype=np.float64).ravel())] * nspan
    flat, spans, o = np.asarray(step_len, dtype=np.float64).ravel(), [], 0
    for n in span_steps:
        spans.append(list(flat[o:o + int(n)]))
        o += int(n)
    return spans


# -------------------------------------------------------------------------------------------------------- PMD replay
def forward_partition(steps, lf, nplates):
    """checkstep replayed on one span's forward steps as matrix_ssfm (and pmx_ctl_next) runs it: zprop accumulated step by
    step, the last step ending at lf.  -> list of {'ntrunk', 'nmem', 'ntot', 'dzb'} in forward order"""
    lcorr = lf / nplates
    out, zprop, dz_miss, ntot = [], 0.0, 0.0, 0
    for j, dz in enumerate(steps):
        dz = float(dz)
        zprop = zprop + dz
        zend = lf if j == len(steps) - 1 else zprop
        dzb, dz_miss, nmem, ntrunk = orc.checkstep(zend, dz, lcorr, dz_miss, ntot)
        out.append({'ntrunk': ntrunk, 'nmem': nmem, 'ntot': ntot, 'dzb': list(dzb)})
        ntot = ntot + ntrunk - nmem
    return out


def reversed_brf(brf):
    """the fiber that undoes brf's PMD: plates last to first, db0 negated (inverse_pmd.m)"""
    return {'db0': -np.asarray(brf['db0'], dtype=np.float64)[::-1], 'theta': np.asarray(brf['theta'], dtype=np.float64)[::-1],
            'epsilon': np.asarray(brf['epsilon'], dtype=np.float64)[::-1]}


def inverse_pmd_chain(ux, uy, brfs, betat, db1, lf, alphalin, gain=None):
    """the pinned inverse_pmd of the spans' fibers (single column), scaled by (exp(alpha*lf/2)/sqrt(gain))^nspan: what
    PMD-aware DBP with xi = 0 and one step per span must give"""
    n = ux.shape[0]
    full = [dict(b, betat=np.asarray(betat).reshape(n, 1), db1=np.asarray(db1).reshape(n, 1), lcorr=lf / len(b['theta']))
            for b in brfs]
    uinv, _ = orc.inverse_pmd_matrix(full, n)
    fx, fy = orc.fft(ux)[:, 0], orc.fft(uy)[:, 0]
    s = (math.exp(0.5 * alphalin * lf) / (math.sqrt(gain) if gain is not None else 1.0)) ** len(brfs)
    return (orc.ifft((uinv[0, 0] * fx + uinv[0, 1] * fy)[:, None]) * s,
            orc.ifft((uinv[1, 0] * fx + uinv[1, 1] * fy)[:, None]) * s)


def scalar_ssfm_steps(u, betat, dzmaxt, dphimaxt, gam, alphalin, nfft, nfc, lf, fls, real=np.float64):
    """orc.scalar_ssfm without the adaptive step (tolflag 0), replayed operation for operation so that its steps can be
    recorded: -> (u, steps in forward order)"""
    R = np.dtype(real).type
    u = np.array(u, dtype=orc._ctype(real), copy=True)
    gam = np.asarray(gam, dtype=np.float64)
    gamrep = np.asarray(gam, dtype=real).reshape(1, -1) * np.ones((nfft, 1), dtype=real)
    dz = float(orc.nextstep(dzmaxt, dphimaxt, gam, alphalin, u, None, False, real))
    halfalpha = 0.5 * alphalin
    zprop, steps = dz, []
    while zprop < lf:
        u = orc.nl_step(alphalin, gamrep, dz, u, nfc, fls[2], fls[3], real)
        u = orc.lin_step(betat * R(dz), u)
        u = u * np.exp(R(-halfalpha * dz))
        steps.append(dz)
        dz = float(orc.nextstep(dzmaxt, dphimaxt, gam, alphalin, u, None, False, real))
        zprop = zprop + dz
    last_step = lf - zprop + dz
    u = orc.nl_step(alphalin, gamrep, last_step, u, nfc, fls[2], fls[3], real)
    u = orc.lin_step(betat * R(last_step), u)
    u = u * np.exp(R(-halfalpha * last_step))
    steps.append(last_step)
    return u, steps


# ------------------------------------------------------------------------------------------------------ one channel
def channel_bins(nfft, shift, decim):
    """the full-grid bins of the M-grid bins 0..M-1 (FFT order): (k - shift) mod nfft for the signed k"""
    M = nfft // decim
    k = np.fft.fftfreq(M, 1.0 / M).round().astype(np.int64)
    return (k - int(shift)) % nfft


def crop(u, bins, decim):
    """[nfft, ...] time samples -> [M, ...]: the channel's bins at baseband, the time samples decimated by decim"""
    return np.fft.ifft(np.fft.fft(u, axis=0)[bins] / decim, axis=0)


def embed(v, bins, nfft, decim):
    """[M, ...] -> [nfft, ...]: the inverse of crop, zeros on every other bin"""
    spec = np.zeros((nfft,) + v.shape[1:], dtype=np.complex128)
    spec[bins] = np.fft.fft(v, axis=0) * decim
    return np.fft.ifft(spec, axis=0)


def band_pass(u, bins):
    """the ideal band-pass onto bins"""
    full = np.fft.fft(u, axis=0)
    spec = np.zeros_like(full)
    spec[bins] = full[bins]
    return np.fft.ifft(spec, axis=0)


def _cut(t, bins):
    """a one-column per-bin table ([nfft] or [nfft, 1]; None stays None) on the channel's bins"""
    return None if t is None else np.asarray(t, dtype=np.float64).reshape(-1, 1)[bins]


# --------------------------------------------------------------------------------------------- nonlinear-step intensity
def gauss_response(nfft, bw):
    """H[k] at the FFT-ordered bins k = 0..nfft-1 (signed bin k_s in [-nfft/2, nfft/2))"""
    ks = np.fft.fftfreq(nfft, 1.0 / nfft)
    return np.exp(-(math.log(2.0) / 2) * (ks / float(bw)) ** 2)


def circular_response(nfft, taps):
    """fft of the taps placed circularly on a grid of nfft samples (c[K] at 0, c[K+m] at m mod nfft): the H with which
    filtered DBP computes the step of the taps"""
    c = np.asarray(taps, dtype=np.float64).ravel()
    k = c.size // 2
    h = np.zeros(nfft)
    for j in range(c.size):
        h[(j - k) % nfft] += c[j]
    return np.fft.fft(h)


def lowpass(q, H):
    """ifft(fft(q) .* H) along the samples of every column"""
    return np.fft.ifft(np.fft.fft(q, axis=0) * H[:, None], axis=0)


def fir(q, taps):
    """the circular FIR of every column of q, summed left to right in the lag m = -K..K (np.roll(q, m)[n] = q[n - m])"""
    c = np.asarray(taps, dtype=np.float64).ravel()
    k = c.size // 2
    out = np.zeros_like(q)
    for j in range(c.size):
        out = out + c[j] * np.roll(q, j - k, axis=0)
    return out


def intensity(nfft, bw=None, taps=None, response=None):
    """the nonlinear-step intensity on an nfft-sample grid: a function (p, s3 or None) -> (p~, s3~ or None), or None for
    plain DBP.  The low-pass filters p + i*s3 as one complex array; the FIR takes p and s3 one after the other."""
    if sum(x is not None for x in (bw, taps, response)) > 1:
        raise ValueError('give at most one of bw, taps and response')
    if taps is not None:
        return lambda p, s3: (fir(p, taps), None if s3 is None else fir(s3, taps))
    if bw is not None:
        response = gauss_response(nfft, bw)
    if response is None:
        return None
    H = np.asarray(response)

    def op(p, s3):
        f = lowpass(p if s3 is None else p + 1j * s3, H)
        return f.real, None if s3 is None else f.imag
    return op


def matrix_nl_step(ismanakov, alphalin, gam, dz, ux, uy, nfc, spm, op, real=np.float64):
    """orc.matrix_nl_step (no xpm) itself for op = None; else with the power and s3 of the field entering the step
    replaced by op's"""
    if op is None:
        return orc.matrix_nl_step(ismanakov, alphalin, gam, dz, ux, uy, nfc, spm, 0, real)
    if not spm:
        return ux, uy
    R = np.dtype(real).type
    leff = orc._leff(alphalin, dz, real)
    p = ux.real ** 2 + ux.imag ** 2 + uy.real ** 2 + uy.imag ** 2
    pf, s3f = op(p, None if ismanakov else 2 * (ux.real * uy.imag - ux.imag * uy.real))
    for k in range(nfc):
        gamleff = R(gam[k]) * leff
        e = orc.fastexp(-gamleff * pf[:, k])
        ux[:, k] = ux[:, k] * e
        uy[:, k] = uy[:, k] * e
        if not ismanakov:
            e = orc.fastexp(gamleff * s3f[:, k] / 3)
            c, s = e.real, e.imag
            ux[:, k], uy[:, k] = c * ux[:, k] + s * uy[:, k], -s * ux[:, k] + c * uy[:, k]
    return ux, uy


def nl_step(alphalin, gam, dz, u, nfc, spm, xpm, op, real=np.float64):
    """orc.nl_step itself for op = None; else with every |u_j|^2 replaced by op's"""
    if op is None:
        return orc.nl_step(alphalin, gam, dz, u, nfc, spm, xpm, real)
    leff = orc._leff(alphalin, dz, real)
    powr = op(u.real ** 2 + u.imag ** 2, None)[0]
    if xpm:
        tot = np.sum(powr, axis=1, keepdims=True) * np.ones((1, nfc), dtype=powr.dtype)
        powr = 2 * tot - powr if spm else 2 * (tot - powr)
    elif not spm:
        return u
    return u * orc.fastexp(-gam * powr * leff)


# ------------------------------------------------------------------------------------------------------- entry points
def dbp(ux, uy, betat, gam, alphalin, nfc, lf, manakov, spm=1, nspan=1, gain=None, steps_per_span=None,
        step_len=None, span_steps=None, xi=1.0, real=np.float64, bw=None, taps=None, response=None):
    """Digital backpropagation (an extension: the reference has no DBP; polmux_ssfm.h, pmx_dbp_desc).  Spans last
    first; for each: u <- u/sqrt(gain), then the span's steps h in reverse of their forward order, each
    u <- exp(+alpha*h/2)*u, u <- lin_step(-betat*h, u) per column, u <- matrix_nl_step with gam -> -xi*gam (the forward
    leff(h), the Manakov 8/9).  Schedule as _spans.  gain: linear amplifier gain after every span, or None.  bw, taps,
    response: the nonlinear-step intensity."""
    return dbp_pmd(ux, uy, betat, None, gam, alphalin, nfc, lf, manakov, None, spm=spm, nspan=nspan, gain=gain,
                   steps_per_span=steps_per_span, step_len=step_len, span_steps=span_steps, xi=xi, real=real, bw=bw,
                   taps=taps, response=response)


def dbp_pmd(ux, uy, betat, db1, gam, alphalin, nfc, lf, manakov, brfs, spm=1, nspan=1, gain=None, steps_per_span=None,
            step_len=None, span_steps=None, xi=1.0, real=np.float64, bw=None, taps=None, response=None):
    """PMD-aware DBP (polmux_ssfm.h, pmx_dbp_desc.pmd).  brfs: nspan plate sets {'db0', 'theta', 'epsilon'} in forward span
    order.  As dbp, with the linear part of a step the inverse of the forward step's trunk product.  brfs = None is dbp
    (db1 unused)."""
    R = np.dtype(real).type
    ct = orc._ctype(real)
    ux = np.array(ux, dtype=ct, copy=True)
    uy = np.array(uy, dtype=ct, copy=True)
    op = intensity(ux.shape[0], bw, taps, response)
    g = -float(xi) * np.asarray(gam, dtype=np.float64)
    if manakov == 'yes':
        g = g * 8 / 9
    nbt = -np.asarray(betat, dtype=real).reshape(ux.shape[0], nfc)
    if brfs is not None:
        nplates = len(brfs[0]['theta'])
        lcorr = lf / nplates
        ndb1 = -np.asarray(db1, dtype=real).reshape(ux.shape[0], nfc)
    spans = _spans(nspan, lf, steps_per_span, step_len, span_steps)
    for k in reversed(range(nspan)):
        if gain is not None:
            a = R(1) / np.sqrt(R(gain))
            ux = ux * a
            uy = uy * a
        if brfs is not None:
            rb = reversed_brf(brfs[k])
            part = forward_partition(spans[k], lf, nplates)
        for j in reversed(range(len(spans[k]))):
            h = spans[k][j]
            a = np.exp(R(0.5 * alphalin * h))
            ux = ux * a
            uy = uy * a
            if brfs is None:
                ux = orc.lin_step(nbt * R(h), ux)
                uy = orc.lin_step(nbt * R(h), uy)
            elif part[j]['ntrunk'] > 0:
                st, ntr = part[j], part[j]['ntrunk']
                first = nplates - (st['ntot'] - st['nmem']) - ntr          # 0-based first plate of the reversed table
                ux, uy = orc.matrix_step(nbt, ndb1, st['dzb'][::-1], ntr, ux, uy, rb, first, 0, lcorr, real)
            ux, uy = matrix_nl_step(manakov == 'yes', alphalin, g, h, ux, uy, nfc, spm, op, real)
    return ux, uy


def dbp_scalar(u, betat, gam, alphalin, nfc, lf, spm=1, xpm=0, nspan=1, gain=None, steps_per_span=None, step_len=None,
               span_steps=None, xi=1.0, real=np.float64, bw=None, taps=None, response=None):
    """Scalar-path DBP.  u: [nfft, nfc] (GSTATE.FIELDX).  Spans last first; for each: u <- u/sqrt(gain), then the span's
    steps h in reverse of their forward order, each u <- exp(+alpha*h/2)*u, u <- lin_step(-betat*h, u), u <- nl_step with
    gam -> -xi*gam (the forward leff(h); with xpm the cross-phase modulation over all columns).  Schedule and intensity as
    dbp."""
    R = np.dtype(real).type
    u = np.array(u, dtype=orc._ctype(real), copy=True)
    nfft = u.shape[0]
    op = intensity(nfft, bw, taps, response)
    g = (-float(xi) * np.asarray(gam, dtype=np.float64)).astype(real).reshape(1, -1) * np.ones((nfft, 1), dtype=real)
    betat = np.asarray(betat, dtype=real).reshape(nfft, nfc)
    spans = _spans(nspan, lf, steps_per_span, step_len, span_steps)
    for k in reversed(range(nspan)):
        if gain is not None:
            u = u * (R(1) / np.sqrt(R(gain)))
        for h in reversed(spans[k]):
            u = u * np.exp(R(0.5 * alphalin * h))
            u = orc.lin_step(-betat * R(h), u)
            u = nl_step(alphalin, g, h, u, nfc, spm, xpm, op, real)
    return u


def dbp_channel(ux, uy, betat, gam, alphalin, lf, manakov, shift, decim, db1=None, brfs=None, spm=1, **kw):
    """Two polarizations, one column ([nfft, 1] each): dbp, or with brfs dbp_pmd, of the channel on nfft/decim samples;
    schedule, xi, gain and intensity as those take them."""
    nfft = ux.shape[0]
    b = channel_bins(nfft, shift, decim)
    vx, vy = dbp_pmd(crop(ux, b, decim), crop(uy, b, decim), _cut(betat, b), _cut(db1, b), gam, alphalin, 1, lf, manakov,
                     brfs, spm=spm, **kw)
    return embed(vx, b, nfft, decim), embed(vy, b, nfft, decim)


def dbp_channel_scalar(u, betat, gam, alphalin, lf, shift, decim, spm=1, **kw):
    """The scalar path, one column ([nfft, 1]): dbp_scalar of the channel on nfft/decim samples; schedule, xi, gain and
    intensity as it takes them."""
    nfft = u.shape[0]
    b = channel_bins(nfft, shift, decim)
    return embed(dbp_scalar(crop(u, b, decim), _cut(betat, b), gam, alphalin, 1, lf, spm=spm, **kw), b, nfft, decim)
