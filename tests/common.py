"""Shared scenario builders: the same seeded Tx field handed to the oracle and to the CUDA path."""
import numpy as np

import oracle.fiber_oracle as orc
import polmux_b200 as pmx
from polmux_b200 import synth
from polmux_b200.fiber import fiber_setup


def base_fiber(**kw):
    f = dict(synth.SMF)
    f['length'] = 8e4
    f.update(kw)
    return f


def make_tx(nsymb, nt, nch=1, rate=28.0, pavg_mw=2.0, ftype='unique', real=np.float64, spac=0.4):
    """-> (oracle GState, fills the product's GSTATE) with identical PDM-QPSK fields."""
    ex, ey, _, _ = synth.pdm_qpsk(nsymb, nt, nch)
    lams = synth.wdm_lambdas(nch, 1550.0, spac)
    power = np.full(nch, float(pavg_mw))
    # oracle side
    gs = orc.reset_all(nsymb, nt, nch, real=real)
    gs.SYMBOLRATE, gs.LAMBDA, gs.POWER = rate, lams.copy(), power.copy()
    orc.create_field(gs, ftype, ex, ey, power_average=True)
    # product side
    pmx.reset_all(nsymb, nt, nch)
    G = pmx.GSTATE
    G.SYMBOLRATE, G.LAMBDA, G.POWER = rate, lams.copy(), power.copy()
    pmx.create_field(ftype, ex, ey, {'power': 'average'})
    return gs


def scalar_tx(nsymb, nt, nch, rate=10.0, pavg=4.0):
    """-> oracle GState; the product's GSTATE holds the same single-polarization field (FIELDY empty), 'sepfields' for
    nch > 1"""
    ex, _, _, _ = synth.pdm_qpsk(nsymb, nt, nch)
    lams = synth.wdm_lambdas(nch, 1550.0, 0.4)
    gs = orc.reset_all(nsymb, nt, nch)
    gs.SYMBOLRATE, gs.LAMBDA, gs.POWER = rate, lams.copy(), np.full(nch, pavg)
    orc.create_field(gs, 'sepfields' if nch > 1 else 'unique', ex, None, power_average=True)
    pmx.reset_all(nsymb, nt, nch)
    G = pmx.GSTATE
    G.SYMBOLRATE, G.LAMBDA, G.POWER = rate, lams.copy(), np.full(nch, pavg)
    pmx.create_field('sepfields' if nch > 1 else 'unique', ex, None, {'power': 'average'})
    return gs


def rel_l2(ux, uy, rx, ry):
    return orc.rel_l2(ux, uy, rx, ry)


def _rel(a, b):
    return float(np.linalg.norm(np.asarray(a) - np.asarray(b)) / np.linalg.norm(np.asarray(b)))


def _cols(a):
    return np.ascontiguousarray(np.asarray(a).T)[None]          # GSTATE [nfft, nfc] -> [1][nfc][nfft]


def _mc_scenario(nsymb, nt, pavg_mw):
    ex, ey, sx, sy = synth.pdm_qpsk(nsymb, nt, 1)
    pmx.reset_all(nsymb, nt, 1)
    G = pmx.GSTATE
    G.SYMBOLRATE, G.LAMBDA, G.POWER = 28.0, np.array([1550.0]), np.array([float(pavg_mw)])
    pmx.create_field('unique', ex, ey, {'power': 'average'})
    fib = dict(synth.SMF)
    fib.update(length=8e4, dgd=0.3, nplates=20, manakov='yes')
    setup = fiber_setup(fib, 'gps-', rng=np.random.Generator(np.random.PCG64(0)))
    return G, setup, np.stack([sx[:, 0], sy[:, 0]]).astype(np.uint8)
