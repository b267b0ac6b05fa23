"""Digital backpropagation restated in numpy (TEST INFRASTRUCTURE): the oracle of pmx_dbp_create / pmx_dbp_exec.

The reference has no DBP, so there is no reference source to pin this against.  It is built from the pinned forward
oracle's own operators -- matrix_nl_step (fiber.m:827-874), lin_step (fiber.m:771-773) and its leff -- in the order
polmux_ssfm.h documents, and tied to the forward oracle by one property that tests/test_dbp.py checks: with the forward
run's own steps, xi = 1 and no noise or PMD, it returns the transmitted field up to rounding.  Like the forward oracle
it is written for a real dtype chosen by the caller.  It is never imported by the product package.
"""
import numpy as np

import oracle.fiber_oracle as orc


def dbp(ux, uy, betat, gam, alphalin, nfc, lf, manakov, spm=1, nspan=1, gain=None, steps_per_span=None,
        step_len=None, span_steps=None, xi=1.0, real=np.float64):
    """Digital backpropagation (an extension: the reference has no DBP; polmux_ssfm.h, pmx_dbp_desc).  Spans last
    first; for each: u <- u/sqrt(gain), then the span's steps h in reverse of their forward order, each
    u <- exp(+alpha*h/2)*u, u <- lin_step(-betat*h, u) per column, u <- matrix_nl_step with gam -> -xi*gam (the forward
    leff(h), the Manakov 8/9).  Schedule: steps_per_span uniform steps of lf/steps_per_span, or step_len -- one span's
    steps for every span, or with span_steps [nspan] all spans' steps concatenated, each span in forward order.
    gain: linear amplifier gain after every span, or None."""
    R = np.dtype(real).type
    ct = orc._ctype(real)
    ux = np.array(ux, dtype=ct, copy=True)
    uy = np.array(uy, dtype=ct, copy=True)
    g = -float(xi) * np.asarray(gam, dtype=np.float64)
    if manakov == 'yes':
        g = g * 8 / 9
    if step_len is None:
        m = int(steps_per_span or 1)
        spans = [[lf / m] * m for _ in range(nspan)]
    elif span_steps is None:
        spans = [list(np.asarray(step_len, dtype=np.float64).ravel())] * nspan
    else:
        flat, spans, o = np.asarray(step_len, dtype=np.float64).ravel(), [], 0
        for n in span_steps:
            spans.append(list(flat[o:o + int(n)]))
            o += int(n)
    betat = np.asarray(betat, dtype=real).reshape(ux.shape[0], nfc)
    for k in reversed(range(nspan)):
        if gain is not None:
            a = R(1) / np.sqrt(R(gain))
            ux = ux * a
            uy = uy * a
        for h in reversed(spans[k]):
            a = np.exp(R(0.5 * alphalin * h))
            ux = ux * a
            uy = uy * a
            ux = orc.lin_step(-betat * R(h), ux)
            uy = orc.lin_step(-betat * R(h), uy)
            ux, uy = orc.matrix_nl_step(manakov == 'yes', alphalin, g, h, ux, uy, nfc, spm, 0, real)
    return ux, uy
