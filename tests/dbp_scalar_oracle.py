"""Digital backpropagation on the scalar path restated in numpy (TEST INFRASTRUCTURE): the oracle of pmx_dbp_create /
pmx_dbp_exec for a field without FIELDY, the scalar counterpart of tests/dbp_oracle.dbp.

Built from the pinned forward oracle's own nl_step (fiber.m:787-804, cross-phase modulation included), lin_step
(fiber.m:771-773) and _leff, in the order polmux_ssfm.h documents.  nl_step is a pure phase per sample and its power
(with 'x': sum_j |u_j|^2 of the sample) depends only on powers, which every step preserves; so with the forward steps and
xi = 1 this oracle inverts scalar_ssfm exactly, XPM included.  tests/test_dbp_small.py checks that property, with the
forward steps replayed by scalar_ssfm_steps (checked there to reproduce scalar_ssfm bit for bit).  Written for a real
dtype chosen by the caller; never imported by the product package.
"""
import numpy as np

import oracle.fiber_oracle as orc


def _spans(nspan, lf, steps_per_span, step_len, span_steps):
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


def dbp_scalar(u, betat, gam, alphalin, nfc, lf, spm=1, xpm=0, nspan=1, gain=None, steps_per_span=None, step_len=None,
               span_steps=None, xi=1.0, real=np.float64):
    """Scalar-path DBP.  u: [nfft, nfc] (GSTATE.FIELDX).  Spans last first; for each: u <- u/sqrt(gain), then the span's
    steps h in reverse of their forward order, each u <- exp(+alpha*h/2)*u, u <- lin_step(-betat*h, u), u <- nl_step with
    gam -> -xi*gam (the forward leff(h); with xpm the cross-phase modulation over all columns).  Schedule as
    dbp_oracle.dbp."""
    R = np.dtype(real).type
    u = np.array(u, dtype=orc._ctype(real), copy=True)
    nfft = u.shape[0]
    g = (-float(xi) * np.asarray(gam, dtype=np.float64)).astype(real).reshape(1, -1) * np.ones((nfft, 1), dtype=real)
    betat = np.asarray(betat, dtype=real).reshape(nfft, nfc)
    spans = _spans(nspan, lf, steps_per_span, step_len, span_steps)
    for k in reversed(range(nspan)):
        if gain is not None:
            u = u * (R(1) / np.sqrt(R(gain)))
        for h in reversed(spans[k]):
            u = u * np.exp(R(0.5 * alphalin * h))
            u = orc.lin_step(-betat * R(h), u)
            u = orc.nl_step(alphalin, g, h, u, nfc, spm, xpm, real)
    return u


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
