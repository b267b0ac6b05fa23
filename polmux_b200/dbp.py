"""dbp(x, flag, ...): digital backpropagation of a link on the received field.

An extension: the reference has no DBP.  The field is run back through a virtual copy of the link -- dispersion,
nonlinearity and loss negated, spans last first, the amplifier gain undone before each span -- on the kernels fiber()
uses for the same field (pmx_dbp_create / pmx_dbp_exec, include/polmux_ssfm.h): the three passes per step for
two-polarization fields of 2^12 to 2^24 samples, the single-launch on-chip kernel (the whole link in one launch) for
smaller fields and for the scalar path (FIELDY empty, 2^6 to 2^12 samples, at most 8 columns).  On the scalar path
with the 'x' flag every step's nonlinear phase includes the cross-phase modulation of all backpropagated columns
(nl_step with gam -> -xi*gam), so a 'sepfields' multiplex is backpropagated as a whole; without 'x' each column is
backpropagated on its own self-phase alone.  With xi = 1 and the forward run's own steps (fiber(..., trace=True) leaves
them in FIBER_LAST['trace_dz']) it inverts a noise-free link without PMD up to rounding; with fewer steps or xi < 1 it is
the receiver-side nonlinear compensation a Monte-Carlo run can count errors behind (McRunner(compensation='dbp')).
Given the link's waveplates (dbp_plan(plates=...), dbp(brf=...)) it is PMD-aware: every step undoes the forward step's
own trunk product as well, so that it inverts a 'gps-' link too (McRunner(compensation='dbp_pmd')).  There is no CPU
fallback.

Single-channel DBP (dbp(..., ich=, decim=), dbp_plan(..., shift=, decim=); pmx_dbp_channel_create): a coherent receiver sees
its own channel only.  Channel ich of a 'unique' multiplex (one column holding every channel) is cut out by an ideal
band-pass, brought to baseband and decimated to nfft/decim samples, backpropagated there on the channel's own dispersion
-- on the route DBP takes for that size -- then interpolated back and returned to its own bins; the other channels are
dropped.  A receiver downstream is unchanged: receiver_cohmix still shifts the channel by its ndfn and filters it.
"""
from __future__ import annotations

from typing import Optional

import numpy as np

from . import _lib
from .fiber import FiberSetup, _get, fiber_setup, setup_to_desc
from .gstate import GSTATE


def dbp_plan(ctx: _lib.Context, setup: FiberSetup, nspan: int = 1, gain_db: Optional[float] = None,
             steps_per_span: Optional[int] = None, step_len=None, span_steps=None, xi: float = 1.0, batch: int = 1,
             precision: Optional[str] = None, disp_mode: Optional[str] = None, plates=None, shift: Optional[int] = None,
             decim: Optional[int] = None, filter_bw: Optional[float] = None, nl_taps=None) -> _lib.DbpPlan:
    """The DBP of nspan spans of the fiber `setup` describes, for resident fields of `batch` realizations.  Schedule:
    steps_per_span uniform steps per span (default 1), or step_len -- one span's steps in forward order for every span,
    or with span_steps [nspan] all spans' steps concatenated.  plates: None -- the 'p' flag, plates and dgdrms are
    ignored; (db0, theta, epsilon), each [nspan][plate_sets][nplates] in forward order (plate_sets 1 or batch) -- PMD-aware
    DBP through those waveplates (setup must carry the 'p' flag; DbpPlan.set_plates swaps in another draw).
    decim: single-channel DBP of a one-column field -- the channel that `shift` bins bring to baseband (the receiver's
    ndfn; default 0), backpropagated on nfft/decim samples (pmx_dbp_channel_create).
    filter_bw [GHz]: filtered DBP -- a Gaussian low-pass of that one-sided -3 dB bandwidth on the intensity of every
    nonlinear step (DbpPlan.set_filter, in bins of GSTATE.FN: filter_bw * NSYMB / SYMBOLRATE); None or 0: none.
    nl_taps: enhanced split-step DBP -- the real circular FIR c[0..2K] (c[K] at lag 0, 2K+1 <= 65 taps) on the intensity of
    every nonlinear step, on the plan's grid (DbpPlan.set_taps; with decim the channel's nfft/decim samples); None or []:
    none.  Not together with filter_bw."""
    taps = _check_taps(nl_taps, filter_bw)
    if plates is not None and not setup.fls[1]:
        raise ValueError("PMD-aware DBP (plates given) needs a fiber with the 'p' flag")
    if decim is None and shift is not None:
        raise ValueError('dbp_plan: shift selects a channel for single-channel DBP and needs decim')
    desc, keep = setup_to_desc(setup, batch=batch, disp_mode=disp_mode, precision=precision)
    gain = 0.0 if gain_db is None else 10 ** (gain_db * 0.1)
    if step_len is None and steps_per_span is None:
        steps_per_span = 1
    d, dkeep = _lib.make_dbp(nspan, gain, steps_per_span=steps_per_span, step_len=step_len, span_steps=span_steps, xi=xi,
                             pmd=plates is not None)
    band = None if decim is None else _lib.make_band(shift or 0, decim)
    plan = _lib.DbpPlan(ctx, desc, keep, d, dkeep, band)
    try:
        if plates is not None:
            arrs = [np.asarray(a, dtype=np.float64).reshape(int(nspan), -1, setup.nplates) for a in plates]
            plan.set_plates(*arrs, plate_sets=arrs[0].shape[1])
        if filter_bw is not None:
            plan.set_filter(float(filter_bw) * GSTATE.NSYMB / GSTATE.SYMBOLRATE)
        if taps.size:
            plan.set_taps(taps)
    except Exception:
        plan.close()
        raise
    return plan


def _check_taps(nl_taps, filter_bw) -> np.ndarray:
    """the taps as float64 (empty: none), refused with pmx_dbp_set_taps's messages before any plan is made"""
    taps = _lib.check_taps(nl_taps)
    if taps.size and filter_bw:
        raise ValueError('pmx_dbp_set_taps: the plan has a filter bandwidth (pmx_dbp_set_filter); a plan takes one or the other')
    return taps


def dbp(x, flag: str, nspan: int = 1, gain_db: Optional[float] = None, steps_per_span: Optional[int] = None, step_len=None,
        span_steps=None, xi: float = 1.0, ctx: Optional[_lib.Context] = None, precision: Optional[str] = None, brf=None,
        ich: Optional[int] = None, decim: Optional[int] = None, filter_bw: Optional[float] = None, nl_taps=None):
    """Backpropagates GSTATE.FIELDX / FIELDY in place through nspan spans of the fiber x, the amplifier of gain_db [dB]
    after each (None: no amplifier).  x and flag are what fiber() takes; a field without FIELDY runs the scalar path, the
    'x' flag there backpropagating the cross-phase modulation of all columns.  Without brf the flag's 'p' is dropped (no plates
    are drawn, nothing is taken from the global random stream) but the fiber's nonlinear model stays the one fiber() used:
    Manakov when x.manakov is 'yes' and the flag has 'p', else the CNLSE.  brf: the struct fiber() returned (every span
    the same plates) or a list of nspan of them in forward span order, with 'p' in the flag: PMD-aware DBP through those
    plates.  xi: fraction of gamma backpropagated.  ich, decim: single-channel DBP of channel ich (1-based) of a 'unique'
    multiplex on nfft/decim samples; afterwards the field holds that channel alone, on its own bins.  filter_bw [GHz]:
    filtered DBP, a Gaussian low-pass of that one-sided -3 dB bandwidth on the intensity of every nonlinear step.  nl_taps:
    enhanced split-step DBP, the real circular FIR c[0..2K] (c[K] at lag 0) on the intensity of every nonlinear step
    (dbp_plan).  The field stays resident on the device like fiber() and ampliflat() leave it."""
    G = GSTATE
    f = str(flag).lower()
    if len(f) != 4:
        raise ValueError("wrong flag. E.g. flag can be 'g---','gp--','-s--', etc")
    _check_taps(nl_taps, filter_bw)
    shift = None
    if decim is not None:
        if ich is None:
            raise ValueError('dbp: single-channel DBP (decim) needs the channel ich')
        if ich < 1 or ich > G.NCH:
            raise ValueError('The channel does not exist')
        if G.field_shape()[1] != 1:
            raise ValueError("dbp: single-channel DBP takes a field holding every channel in one column ('unique')")
        from .receiver import channel_ndfn
        shift = int(channel_ndfn(ich, G)) if G.NCH > 1 else 0
    elif ich is not None:
        raise ValueError('dbp: ich selects a channel for single-channel DBP and needs decim')
    plates = None
    if brf is None:
        s = fiber_setup(x, f[0] + '-' + f[2:])
    else:
        if f[1] != 'p':
            raise ValueError("dbp: brf (PMD-aware DBP) needs the 'p' flag")
        # (a private stream: the plates come from brf, nothing is drawn from the global one)
        s = fiber_setup(x, f, rng=np.random.Generator(np.random.PCG64(0)))
        brfs = [brf] * int(nspan) if isinstance(brf, dict) else list(brf)
        if len(brfs) != int(nspan):
            raise ValueError('dbp: brf must be one struct or a list of nspan of them')
        for b in brfs:
            if np.asarray(b['theta']).size != s.nplates:
                raise ValueError('dbp: brf has %d plates, the fiber %d' % (np.asarray(b['theta']).size, s.nplates))
        plates = tuple(np.stack([np.asarray(b[k], dtype=np.float64).reshape(1, -1) for b in brfs])
                       for k in ('db0', 'theta', 'epsilon'))
    if s.fls[3] and s.isv:
        raise NotImplementedError('The CNLSE with separate fields is not yet implemented')    # fiber.m:854
    if s.isv and not G.has_y():                                  # the 'p' flag on a single-polarization field (:285-289)
        G.FIELDY = np.zeros_like(G.FIELDX)
    s.manakov = f[1] == 'p' and str(_get(x, 'manakov', 'no')) == 'yes'
    ctx = ctx or _lib.default_context()
    from .fiber import PRECISION                                 # (the module default, read at call time)
    prec = {'f64': _lib.PMX_F64, 'f32': _lib.PMX_F32}[precision or PRECISION]
    if not s.isv:
        # scalar path: host buffers like the scalar fiber() -- upload, plan, execute, download into FIELDX
        fx = np.ascontiguousarray(np.asarray(G.FIELDX, dtype=np.complex128).T)[None]     # [1][nfc][nfft]
        fld = _lib.DeviceField(ctx, s.nfft, s.nfc, 1, precision=prec)
        try:
            fld.upload(fx, np.zeros_like(fx))
            plan = dbp_plan(ctx, s, nspan, gain_db, steps_per_span, step_len, span_steps, xi, precision=precision,
                            shift=shift, decim=decim, filter_bw=filter_bw, nl_taps=nl_taps)
            try:
                plan.execute(fld)
            finally:
                plan.close()
            ux, _ = fld.download()
        finally:
            fld.close()
        G.FIELDX = np.ascontiguousarray(ux[0].T)
        return
    fld, hx, hy = G.take_device(ctx, prec)
    try:
        plan = dbp_plan(ctx, s, nspan, gain_db, steps_per_span, step_len, span_steps, xi, precision=precision, plates=plates,
                        shift=shift, decim=decim, filter_bw=filter_bw, nl_taps=nl_taps)
    except Exception:
        G.restore_host(fld, hx, hy)     # nothing ran: the caller's field is as it was
        raise
    try:
        plan.execute(fld)
    except Exception:
        fld.close()                     # part-way through the link: not usable
        raise
    finally:
        plan.close()
    G.put_device(fld, hx, hy)
