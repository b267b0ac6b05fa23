"""PMD-aware digital backpropagation restated in numpy (TEST INFRASTRUCTURE): the oracle of pmx_dbp_create with pmd = 1.

Built from the pinned forward oracle's own checkstep (fiber.m:739-758), matrix_step (fiber.m:904-935), matrix_nl_step
(fiber.m:827-874) and _leff.  A DBP step undoes the forward step: its trunk pieces are the forward run's, replayed from
the forward steps (forward_partition), and the linear step is a forward matrix_step of the reversed fiber -- plates
last to first, db0, db1 and betat negated, the pieces mirrored.  tests/test_dbp_pmd.py ties it to the forward oracle
(with the forward steps and xi = 1 it returns the Tx field) and to the pinned inverse_pmd (xi = 0, one step per span).
It is never imported by the product package.
"""
import math

import numpy as np

import oracle.fiber_oracle as orc


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


def dbp_pmd(ux, uy, betat, db1, gam, alphalin, nfc, lf, manakov, brfs, spm=1, nspan=1, gain=None, steps_per_span=None,
            step_len=None, span_steps=None, xi=1.0, real=np.float64):
    """PMD-aware DBP (polmux_ssfm.h, pmx_dbp_desc.pmd).  brfs: nspan plate sets {'db0', 'theta', 'epsilon'} in forward span
    order.  Spans last first; for each: u <- u/sqrt(gain), then the span's steps h in reverse of their forward order, each
    u <- exp(+alpha*h/2)*u, the inverse of the forward step's trunk product, matrix_nl_step with gam -> -xi*gam.
    Schedule as dbp_oracle.dbp."""
    R = np.dtype(real).type
    ct = orc._ctype(real)
    ux = np.array(ux, dtype=ct, copy=True)
    uy = np.array(uy, dtype=ct, copy=True)
    g = -float(xi) * np.asarray(gam, dtype=np.float64)
    if manakov == 'yes':
        g = g * 8 / 9
    nplates = len(brfs[0]['theta'])
    lcorr = lf / nplates
    nbt = -np.asarray(betat, dtype=real).reshape(ux.shape[0], nfc)
    ndb1 = -np.asarray(db1, dtype=real).reshape(ux.shape[0], nfc)
    spans = _spans(nspan, lf, steps_per_span, step_len, span_steps)
    for k in reversed(range(nspan)):
        if gain is not None:
            a = R(1) / np.sqrt(R(gain))
            ux = ux * a
            uy = uy * a
        rb = reversed_brf(brfs[k])
        part = forward_partition(spans[k], lf, nplates)
        for h, st in zip(reversed(spans[k]), reversed(part)):
            a = np.exp(R(0.5 * alphalin * h))
            ux = ux * a
            uy = uy * a
            ntr = st['ntrunk']
            first = nplates - (st['ntot'] - st['nmem']) - ntr          # 0-based first plate of the reversed table
            if ntr > 0:
                ux, uy = orc.matrix_step(nbt, ndb1, st['dzb'][::-1], ntr, ux, uy, rb, first, 0, lcorr, real)
            ux, uy = orc.matrix_nl_step(manakov == 'yes', alphalin, g, h, ux, uy, nfc, spm, 0, real)
    return ux, uy


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
