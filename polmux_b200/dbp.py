"""dbp(x, flag, ...): digital backpropagation of a link on the received field.

An extension: the reference has no DBP.  The field is run back through a virtual copy of the link -- dispersion,
nonlinearity and loss negated, spans last first, the amplifier gain undone before each span -- on the same three-pass
kernels as fiber() (pmx_dbp_create / pmx_dbp_exec, include/polmux_ssfm.h).  With xi = 1 and the forward run's own
steps (fiber(..., trace=True) leaves them in FIBER_LAST['trace_dz']) it inverts a noise-free link without PMD up to
rounding; with fewer steps or xi < 1 it is the receiver-side nonlinear compensation a Monte-Carlo run can count errors
behind (McRunner(compensation='dbp')).  There is no CPU fallback.
"""
from __future__ import annotations

from typing import Optional

from . import _lib
from .fiber import FiberSetup, _get, fiber_setup, setup_to_desc
from .gstate import GSTATE


def dbp_plan(ctx: _lib.Context, setup: FiberSetup, nspan: int = 1, gain_db: Optional[float] = None,
             steps_per_span: Optional[int] = None, step_len=None, span_steps=None, xi: float = 1.0, batch: int = 1,
             precision: Optional[str] = None, disp_mode: Optional[str] = None) -> _lib.DbpPlan:
    """The DBP of nspan spans of the fiber `setup` describes (its 'p' flag, plates and dgdrms are ignored), for resident
    fields of `batch` realizations.  Schedule: steps_per_span uniform steps per span (default 1), or step_len -- one
    span's steps in forward order for every span, or with span_steps [nspan] all spans' steps concatenated."""
    desc, keep = setup_to_desc(setup, batch=batch, disp_mode=disp_mode, precision=precision)
    gain = 0.0 if gain_db is None else 10 ** (gain_db * 0.1)
    if step_len is None and steps_per_span is None:
        steps_per_span = 1
    d, dkeep = _lib.make_dbp(nspan, gain, steps_per_span=steps_per_span, step_len=step_len, span_steps=span_steps, xi=xi)
    return _lib.DbpPlan(ctx, desc, keep, d, dkeep)


def dbp(x, flag: str, nspan: int = 1, gain_db: Optional[float] = None, steps_per_span: Optional[int] = None, step_len=None,
        span_steps=None, xi: float = 1.0, ctx: Optional[_lib.Context] = None, precision: Optional[str] = None):
    """Backpropagates GSTATE.FIELDX / FIELDY in place through nspan spans of the fiber x, the amplifier of gain_db [dB]
    after each (None: no amplifier).  x and flag are what fiber() takes; the flag's 'p' is dropped (no plates are drawn,
    nothing is taken from the global random stream) but the fiber's nonlinear model stays the one fiber() used: Manakov
    when x.manakov is 'yes' and the flag has 'p', else the CNLSE.  xi: fraction of gamma backpropagated.
    The field stays resident on the device like fiber() and ampliflat() leave it."""
    G = GSTATE
    f = str(flag).lower()
    if len(f) != 4:
        raise ValueError("wrong flag. E.g. flag can be 'g---','gp--','-s--', etc")
    s = fiber_setup(x, f[0] + '-' + f[2:])
    if not (s.isv and G.has_y()):
        raise NotImplementedError('dbp: two-polarization fields only (the scalar path has no DBP)')
    if s.fls[3]:
        raise NotImplementedError('The CNLSE with separate fields is not yet implemented')    # fiber.m:854
    s.manakov = f[1] == 'p' and str(_get(x, 'manakov', 'no')) == 'yes'
    ctx = ctx or _lib.default_context()
    from .fiber import PRECISION                                 # (the module default, read at call time)
    prec = {'f64': _lib.PMX_F64, 'f32': _lib.PMX_F32}[precision or PRECISION]
    fld, hx, hy = G.take_device(ctx, prec)
    try:
        plan = dbp_plan(ctx, s, nspan, gain_db, steps_per_span, step_len, span_steps, xi, precision=precision)
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
