"""pbnlc(x, flag, ...): perturbation-based nonlinearity compensation (PB-NLC) of a single-channel received field.

An extension: the reference has none.  The first-order regular-perturbation term of the link is written as a sum of
symbol triplets (Mecozzi, Clausen & Shtaif, IEEE PTL 12(4), 2000),

    Delta^x_k = -j*gamma * sum_{m,n} C[m,n] * ( a*A^x_{k+m} A^x_{k+n} conj(A^x_{k+m+n})
                                              + b*A^x_{k+m} A^y_{k+n} conj(A^y_{k+m+n})
                                              + c*A^y_{k+m} A^y_{k+n} conj(A^x_{k+m+n}) )      (x <-> y for Y)

and subtracted at the receiver from the received samples, scaled by xi (Tao et al., JLT 29(17), 2011).  A_k = <p_k, u> is
the field projected onto the pulse of symbol k (centred at time index k*nt, circular over the block).  The weights are
those of the library's nonlinear step: Manakov (1, 1, 0) with gam carrying the 8/9, the CNLSE (1, 2/3, 1/3) -- the
first-order expansion of -j*gam*[P*u + (s3/3)*J*u] (fiber.m:827-851).

The coefficient table C[m,n] of the whole link (pb_coefficients) is computed once, on the host (numpy, the reference) or,
with table='device', by the library (pmx_pb_table: the same table, the lag sums on the device); the stage itself runs on
the device in one pass at the symbol rate (pmx_pb_create / pmx_pb_exec, include/polmux_ssfm.h).  There is no CPU fallback.

Single-channel PB-NLC (pbnlc(..., ich=, decim=), pb_plan(..., shift=, decim=); pmx_pb_channel_create): a coherent receiver
sees its own channel only.  As single-channel DBP does it, channel ich of a 'unique' multiplex is cut out by an ideal
band-pass, brought to baseband and decimated to nfft/decim samples, compensated there with the table of its own dispersion
(channel_setup) and the pulse it carries at that rate (channel_pulse), then returned to its own bins; the other channels
are dropped.

XPM-aware single-channel PB-NLC (pbnlc(..., ich=, decim=, xpm=), pb_plan(..., xpm=); pmx_pb_xpm_create): with the
neighbours' projected symbols B (a joint multi-channel receiver has them), the first-order inter-channel term of each
interferer c in the same triplet form,

    Delta^x_k += -j*gamma * sum_{m,n} D_c[m,n] * ( w1*A^x_{k+m} B^x_{k+n} conj(B^x_{k+m+n}) + w2*A^x_{k+m} B^y_{k+n} conj(B^y_{k+m+n})
                                                 + w3*A^y_{k+m} B^x_{k+n} conj(B^y_{k+m+n}) + w4*A^y_{k+m} B^y_{k+n} conj(B^x_{k+m+n}) )

(x <-> y for Y): the terms of the nonlinear step at the channel's frequency linear in A and in B*conj(B), Manakov (2, 1, 1, 0)
and the CNLSE (2, 2/3, 2/3, 2/3).  D_c (xpm_coefficients) is the overlap of the channel's pulse with the interferer's, each
dispersed with its own dispersion in the channel's frame, so that the interferer keeps its walk-off.  Left out: four-wave
mixing between two interferers and the triplets whose indices do not satisfy i + j - l = k.
"""
from __future__ import annotations

import dataclasses
import math
from typing import Optional

import numpy as np
import scipy.fft as _sfft

from . import _lib
from . import synth
from .fiber import FiberSetup, _get, fiber_setup
from .gstate import GSTATE

# model weights (a, b, c) of the triplet sum
MANAKOV = (1.0, 1.0, 0.0)
CNLSE = (1.0, 2.0 / 3.0, 1.0 / 3.0)
# model weights (w1, w2, w3, w4) of the XPM triplet sum
MANAKOV_XPM = (2.0, 1.0, 1.0, 0.0)
CNLSE_XPM = (2.0, 2.0 / 3.0, 2.0 / 3.0, 2.0 / 3.0)


def model_weights(setup: FiberSetup):
    """(a, b, c) and the gamma of the triplet sum for the nonlinear model the fiber's nonlinear step uses"""
    gam = float(np.asarray(setup.gam, dtype=np.float64).ravel()[0])
    return (MANAKOV, gam * 8 / 9) if setup.manakov else (CNLSE, gam)


def xpm_weights(setup: FiberSetup):
    """(w1, w2, w3, w4) and the gamma of the XPM triplet sum for the nonlinear model the fiber's nonlinear step uses"""
    w, gam = model_weights(setup)
    return (MANAKOV_XPM if setup.manakov else CNLSE_XPM), gam


def pb_nodes(length: float, nspan: int, alphalin: float, nquad: int):
    """Gauss-Legendre nodes of every span -> (accumulated distance zeta [nspan*nquad], weight * exp(-alpha*z))"""
    x, w = np.polynomial.legendre.leggauss(int(nquad))
    z = 0.5 * length * (x + 1.0)
    wz = 0.5 * length * w * np.exp(-alphalin * z)
    zeta = np.concatenate([s * length + z for s in range(int(nspan))])
    return zeta, np.tile(wz, int(nspan))


def _lin_step(betaxdz, u):
    """fiber.m:771-773: ifft(fft(u) .* exp(-i*betaxdz))"""
    return _sfft.ifft(_sfft.fft(u) * (np.cos(betaxdz) - 1j * np.sin(betaxdz)))


def default_window(setup: FiberSetup, nspan: int, pulse, nt: int, K: int, tol: float = 1e-9) -> int:
    """The symbols of the circular window the table is computed on: the smallest power of two that holds the pulse
    dispersed over the whole link (all but `tol` of its energy) plus the 2K symbols of the shifts, at most the block."""
    N = setup.nfft
    nsymb = N // nt
    p0 = np.zeros(N, dtype=np.complex128)
    p0[(np.arange(len(pulse)) - len(pulse) // 2) % N] = pulse
    g = _lin_step(np.asarray(setup.betat, dtype=np.float64)[:, 0] * (setup.length * nspan), p0)
    e = np.abs(np.fft.fftshift(g)) ** 2
    c = np.cumsum(e) / e.sum()
    lo, hi = np.searchsorted(c, 0.5 * tol), np.searchsorted(c, 1 - 0.5 * tol)
    need = (hi - lo + 1) / nt + 2 * K + 8
    w = 1
    while w < need:
        w *= 2
    return int(min(w, nsymb))


def pb_coefficients(setup: FiberSetup, nspan: int, pulse=None, K: int = 16, prune: float = 0.0, nt: Optional[int] = None,
                    nquad: int = 32, window: Optional[int] = None, ctx: Optional[_lib.Context] = None):
    """The triplet coefficients of nspan spans of the fiber `setup` describes:
        C[m,n] = sum_s int_0^Ls exp(-alpha*z) <g_0, g_m g_n conj(g_{m+n})>(s*Ls + z) dz,   |m|, |n| <= K,
    g_m(zeta) the pulse of symbol m (centred at m*nt) after lin_step(betat*zeta) (no loss), <u, v> = sum conj(u) v / sum p^2.
    pulse: default synth.cosroll_pulse(nt, 0.2); nt: default GSTATE.NT.  nquad Gauss-Legendre nodes per span; the table is
    computed on a circular window of `window` symbols (default_window; the link's frequency grid subsampled, so betat is
    the link's own).  prune drops entries with |C| < prune*|C[0,0]|.
    By translation invariance the row m is the autocorrelation of a_m = conj(g_0) g_m at symbol-spaced lags,
    C[m,n] = sum_t a_m(t) conj(a_m(t - n*nt)): one FFT per row and node.  Only the rows m >= 0 are transformed: the
    autocorrelation gives C[m,-n] = conj(C[m,n]), and with C[m,n] = C[n,m], C[-m,n] = conj(C[m,n]).
    ctx: the library computes the same table on that context's device (pmx_pb_table), orders of magnitude faster.
    -> (m, n, C): int32 [ncoef], int32 [ncoef], complex128 [ncoef], m-major with n ascending."""
    nt = int(nt or GSTATE.NT)
    K = int(K)
    if K < 0:
        raise ValueError('pb_coefficients: K must be >= 0')
    p = np.asarray(synth.cosroll_pulse(nt, 0.2) if pulse is None else pulse, dtype=np.float64).ravel()
    if ctx is not None:
        return pb_table(ctx, setup, nspan, p, K, prune, nt, nquad, window)[:3]
    N = int(setup.nfft)
    nsymb = N // nt
    W = int(window or default_window(setup, nspan, p, nt, K))
    if nsymb % W or W < 1:
        raise ValueError('pb_coefficients: the window (%d symbols) must divide the block (%d symbols)' % (W, nsymb))
    Ws = W * nt
    bt = np.asarray(setup.betat, dtype=np.float64)[:, 0][::N // Ws]      # the link's bins that fall on the window's grid
    p0 = np.zeros(Ws, dtype=np.complex128)
    p0[(np.arange(p.size) - p.size // 2) % Ws] = p
    norm = float(np.sum(p * p))
    zeta, wq = pb_nodes(setup.length, nspan, setup.alphalin, nquad)
    spec = np.zeros((K + 1, W))                                            # sum_nodes w * (|fft a_m|^2 folded to W bins)
    for z, w in zip(zeta, wq):
        g0 = _lin_step(bt * z, p0)
        a = np.conj(g0)[None, :] * np.stack([np.roll(g0, m * nt) for m in range(K + 1)])
        s = np.abs(_sfft.fft(a, axis=1)) ** 2
        spec += w * s.reshape(K + 1, nt, W).sum(axis=1)
    row = _sfft.ifft(spec / nt, axis=1) / norm                            # [m >= 0][lag n mod W]
    lags = np.arange(-K, K + 1)
    C = np.empty((2 * K + 1, 2 * K + 1), dtype=np.complex128)
    C[K:, :] = row[:, lags % W]
    C[:K, :] = np.conj(row[1:, lags % W][::-1])
    C = 0.5 * (C + C.T)                                                    # exactly symmetric
    mm, nn = np.meshgrid(lags, lags, indexing='ij')
    keep = np.abs(C) >= float(prune) * abs(C[K, K]) if prune else np.ones(C.shape, dtype=bool)
    return mm[keep].astype(np.int32), nn[keep].astype(np.int32), C[keep]


def pb_table(ctx: Optional[_lib.Context], setup: FiberSetup, nspan: int, pulse, K: int = 16, prune: float = 0.0,
             nt: Optional[int] = None, nquad: int = 32, window: Optional[int] = None):
    """pb_coefficients computed by the library (pmx_pb_table) -> (m, n, C, window): the table and the window it used, in
    symbols (default_window's for window None).  ctx None only checks the arguments, as the library does before it needs a
    device.  A bad argument raises ValueError with the library's message, as the host path raises ValueError for its own."""
    nt = int(nt or GSTATE.NT)
    bt = np.asarray(setup.betat, dtype=np.float64)[:, 0] if np.ndim(setup.betat) == 2 else setup.betat
    try:
        return _lib.pb_table(ctx, _lib.make_pb_table(setup.nfft, nt, bt, pulse, nspan, setup.length, setup.alphalin, K,
                                                     nquad, window, prune))
    except _lib.PolmuxError as e:
        if e.code == _lib.PMX_ERR_INVALID:
            raise ValueError(str(e)) from e
        raise


def _check_table(table: str) -> str:
    if table not in ('host', 'device'):
        raise ValueError("pb_plan: table must be 'host' (numpy) or 'device' (pmx_pb_table), got %r" % (table,))
    return table


def _check_decim(decim, nt: Optional[int] = None) -> int:
    """ValueError with pmx_pb_channel_create's message for a decimation it refuses, and for one that does not divide the
    samples per symbol nt (the channel keeps every symbol), before any table is computed"""
    r = int(decim)
    if r < 2 or r & (r - 1):
        raise ValueError('pmx_pb_channel_create: decim=%d, must be a power of two >= 2' % r)
    if nt is not None and int(nt) % r:
        raise ValueError('decim=%d must divide nt=%d: the channel keeps every symbol at nt/decim samples' % (r, int(nt)))
    return r


def _channel_bins(nfft: int, shift: int, decim: int) -> np.ndarray:
    """the nfft-grid bins of the M = nfft/decim grid's bins 0..M-1 (FFT order): (k - shift) mod nfft for the signed k"""
    M = nfft // decim
    k = np.fft.fftfreq(M, 1.0 / M).round().astype(np.int64)
    return (k - int(shift)) % nfft


def channel_setup(setup: FiberSetup, shift: int, decim: int) -> FiberSetup:
    """The FiberSetup of the channel that `shift` bins bring to baseband (the receiver's ndfn), on M = nfft/decim samples:
    the channel's own dispersion, betat_M[k] = betat_N[(k - shift) mod N] for the signed k of the M grid (db1 likewise),
    the mapping single-channel DBP uses (pmx_dbp_channel_create), less its constant and linear part in k (taken from bins
    0 and +-1).  That part is the channel's phase and group delay, which cancel in conj(g_0) g_m g_n conj(g_{m+n}) as they
    would in continuous time.  On the circular grid they would not quite: a group delay of a fraction of a sample moves
    the table with the aliased part of the products, and a walk-off over the link spreads the pulse over the whole window
    (default_window).  pb_coefficients on this setup is the channel's table; it differs from the centre channel's only
    with a dispersion slope."""
    r = _check_decim(decim)
    N = int(setup.nfft)
    M = N // r
    b = _channel_bins(N, shift, r)
    bt = np.asarray(setup.betat, dtype=np.float64)[b]
    k = np.fft.fftfreq(M, 1.0 / M).round().reshape(-1, 1)
    bt = bt - bt[0] - k * (0.5 * (bt[1] - bt[M - 1]))
    return dataclasses.replace(setup, nfft=M, betat=np.ascontiguousarray(bt),
                               db1=np.ascontiguousarray(np.asarray(setup.db1)[b]))


def channel_pulse(nt: int, decim: int, nfft: int) -> np.ndarray:
    """The default pulse of single-channel PB-NLC at nt/decim samples per symbol: the transmit pulse synth.cosroll_pulse(nt,
    0.2), placed on nfft samples as symbol 0, through the ideal band-pass and decimation of the down step (the real part:
    the band's one unpaired bin -M/2 is split between -M/2 and +M/2), truncated to the 16*nt/decim samples (at most
    nfft/decim) pmx_pb_desc allows, symbol 0 at index npulse/2 as the stage places it.  A model choice: the pulse the field
    carries at that rate, not the pulse a transmitter at that rate would send; pb_plan(pulse=) takes another."""
    r = _check_decim(decim)
    N, M, ntm = int(nfft), int(nfft) // r, int(nt) // r
    p = synth.cosroll_pulse(int(nt), 0.2)
    u = np.zeros(N, dtype=np.complex128)
    u[(np.arange(p.size) - p.size // 2) % N] = p
    v = _sfft.ifft(_sfft.fft(u)[_channel_bins(N, 0, r)] / r).real       # v[n] = (band-passed u)[n*r]
    L = min(16 * ntm, M)
    return np.ascontiguousarray(v[(np.arange(L) - L // 2) % M])


def _frame_betat(setup: FiberSetup, shift: int, ref: int, k) -> np.ndarray:
    """the dispersion per metre of the channel that `shift` bins bring to baseband, at the signed link-grid offsets k from
    its centre, in the frame of the channel at `ref`: betat[(k - shift) mod N] less the channel's constant phase and less
    k times the group delay of channel `ref` (channel_setup's, taken from its bins +-1).  For shift == ref it is
    channel_setup's dispersion; for another channel the walk-off against `ref` stays."""
    N = int(setup.nfft)
    bt = np.asarray(setup.betat, dtype=np.float64).reshape(N, -1)[:, 0]
    k = np.asarray(k, dtype=np.int64)
    c0 = 0.5 * (bt[(1 - int(ref)) % N] - bt[(-1 - int(ref)) % N])
    return bt[(k - int(shift)) % N] - bt[(-int(shift)) % N] - k * c0


def xpm_walkoff(setup: FiberSetup, nspan: int, shift: int, shift_int: int, nt: int) -> float:
    """the walk-off [symbols] of the channel at shift_int against the channel at shift over nspan spans: the difference of
    their group delays (the slopes of betat at their centres) times the length"""
    N = int(setup.nfft)
    c = [0.5 * (_frame_betat(setup, s, 0, [1]) - _frame_betat(setup, s, 0, [-1]))[0] for s in (shift, shift_int)]
    return float((c[1] - c[0]) * setup.length * int(nspan) * N / (2 * math.pi) / int(nt))


def default_xpm_kn(setup: FiberSetup, nspan: int, shift: int, shift_int: int, nt: int, K: int) -> int:
    """|n| <= Kn of an XPM table: K plus the walk-off of the link in symbols plus 8, at most PMX_PB_XPM_MAX_N and half the
    block"""
    w = abs(xpm_walkoff(setup, nspan, shift, shift_int, nt))
    return int(min(int(K) + math.ceil(w) + 8, _lib.PB_XPM_MAX_N, int(setup.nfft) // int(nt) // 2))


def default_xpm_window(setup: FiberSetup, nspan: int, shift: int, shift_int: int, decim: int, pulse, nt: int, K: int,
                       Kn: int) -> int:
    """The symbols of the circular window an XPM table is computed on: the smallest power of two that holds, in the COI's
    frame, the pulse (its npulse samples at nt/decim per symbol) spread by the group delays of the channel's band over the
    link, the same for the interferer's band (its walk-off included, from the start of the link to its end), the K symbols
    of the shifts and the Kn lags, plus 16 -- at most the block.  (An energy rule as default_window's is no use here: the
    band-limited pulse's sinc tails fill the block.)"""
    N, r = int(setup.nfft), int(decim)
    M = N // r
    k = np.fft.fftfreq(M, 1.0 / M).round().astype(np.int64)
    L = setup.length * int(nspan)
    sym = N / (2 * math.pi) / int(nt)                                     # group delay per (rad/bin) in symbols

    def delays(sh):
        gd = np.diff(_frame_betat(setup, sh, shift, np.sort(k))) * L * sym
        return min(0.0, float(gd.min())), max(0.0, float(gd.max()))
    half = 0.5 * len(pulse) / (int(nt) // r)
    g0, g1 = delays(shift)
    h0, h1 = delays(shift_int)
    lo = min(g0, h0 - Kn) - half
    hi = max(g1 + K, h1 + K + Kn) + half
    need = hi - lo + 16
    w = 1
    while w < need:
        w *= 2
    return int(min(w, N // int(nt)))


def xpm_coefficients(setup: FiberSetup, nspan: int, shift: int, shift_int: int, decim: int, pulse=None, K: int = 16,
                     Kn: Optional[int] = None, prune: float = 0.0, nt: Optional[int] = None, nquad: int = 32,
                     window: Optional[int] = None, up: int = 4):
    """The XPM triplet coefficients of the interferer that shift_int bins bring to baseband on the channel at `shift`
    (single-channel PB-NLC at nfft/decim samples, nt/decim samples per symbol; setup the link at nfft samples):
        D[m,n] = sum_s int_0^Ls exp(-alpha*z) <g_0, g_m h_n conj(h_{m+n})>(s*Ls + z) dz,   |m| <= K, |n| <= Kn,
    g_m the channel's pulse of symbol m and h_m the interferer's, each dispersed (lin_step) with its own dispersion in the
    channel's frame (_frame_betat: the interferer keeps its walk-off), <u, v> = sum conj(u) v / sum p^2 at nt/decim samples
    per symbol.  pulse: default channel_pulse (at nt/decim); nt: default GSTATE.NT (the link's); Kn: default_xpm_kn.
    The pulses are band-limited: the pulse's spectrum on the window's grid is zero-padded to `up` times its rate (the
    unpaired bin split between +-half), so that the four-pulse products do not alias (at nt/decim samples per symbol a
    fractional-sample walk-off would move the table with the aliased part).  The window (default_xpm_window) holds `window`
    symbols of the COI's grid.  prune drops entries with |D| < prune*max|D|.
    FFT form: with b_m = conj(g_0) g_m and e_m = conj(h_0) h_m, D[m,n] = sum_t b_m(t) conj(e_m(t - n*nt)), a
    cross-correlation, one FFT pair per row and node; D[-m,n] = conj(D[m,n]), so the rows m >= 0 are transformed.  There is
    no m <-> n symmetry.  -> (m, n, D): int32, int32, complex128 [ncoef], m-major with n ascending."""
    nt = int(nt or GSTATE.NT)
    r = _check_decim(decim, nt)
    K, up = int(K), int(up)
    if K < 0 or K > _lib.PB_MAX_K:
        raise ValueError('xpm_coefficients: K=%d, 0 to %d' % (K, _lib.PB_MAX_K))
    if up < 1:
        raise ValueError('xpm_coefficients: up must be >= 1')
    N = int(setup.nfft)
    ntm, nsymb = nt // r, N // nt
    p = np.asarray(channel_pulse(nt, r, N) if pulse is None else pulse, dtype=np.float64).ravel()
    Kn = int(default_xpm_kn(setup, nspan, shift, shift_int, nt, K) if Kn is None else Kn)
    if Kn < 0 or Kn > _lib.PB_XPM_MAX_N:
        raise ValueError('xpm_coefficients: Kn=%d, 0 to %d' % (Kn, _lib.PB_XPM_MAX_N))
    W = int(window or default_xpm_window(setup, nspan, shift, shift_int, r, p, nt, K, Kn))
    if W < 1 or nsymb % W or 2 * Kn >= W:
        raise ValueError('xpm_coefficients: the window (%d symbols) must divide the block (%d symbols) and exceed 2*Kn = %d'
                         % (W, nsymb, 2 * Kn))
    Wm, ntu = W * ntm, up * ntm
    Ws = up * Wm                                                           # samples of the fine window
    p0 = np.zeros(Wm, dtype=np.complex128)
    p0[(np.arange(p.size) - p.size // 2) % Wm] = p
    P = _sfft.fft(p0)
    k = np.fft.fftfreq(Ws, 1.0 / Ws).round().astype(np.int64)           # signed bins of the fine window
    inb = np.abs(k) <= Wm // 2
    F = np.zeros(Ws, dtype=np.complex128)
    F[inb] = P[k[inb] % Wm]
    F[np.abs(k) == Wm // 2] *= 0.5                                         # the unpaired bin, split between +-Wm/2
    F *= up
    step = nsymb // W                                                      # link bins per window bin
    bg, bh = np.zeros(Ws), np.zeros(Ws)
    bg[inb] = _frame_betat(setup, shift, shift, k[inb] * step)
    bh[inb] = _frame_betat(setup, shift_int, shift, k[inb] * step)
    norm = float(np.sum(p * p)) * up                                       # (the fine sums hold up samples per coarse one)
    zeta, wq = pb_nodes(setup.length, nspan, setup.alphalin, nquad)
    spec = np.zeros((K + 1, W), dtype=np.complex128)
    for z, w in zip(zeta, wq):
        g0 = _sfft.ifft(F * (np.cos(bg * z) - 1j * np.sin(bg * z)))
        h0 = _sfft.ifft(F * (np.cos(bh * z) - 1j * np.sin(bh * z)))
        b = np.conj(g0)[None, :] * np.stack([np.roll(g0, m * ntu) for m in range(K + 1)])
        e = np.conj(h0)[None, :] * np.stack([np.roll(h0, m * ntu) for m in range(K + 1)])
        S = _sfft.fft(b, axis=1) * np.conj(_sfft.fft(e, axis=1))
        spec += w * S.reshape(K + 1, ntu, W).sum(axis=1)
    row = _sfft.ifft(spec / ntu, axis=1) / norm                           # [m >= 0][lag n mod W]
    lags = np.arange(-Kn, Kn + 1)
    D = np.empty((2 * K + 1, 2 * Kn + 1), dtype=np.complex128)
    D[K:, :] = row[:, lags % W]
    D[K, :] = D[K, :].real                                                 # sum |g_0|^2 |h_n|^2: real
    D[:K, :] = np.conj(row[1:, lags % W][::-1])
    mm, nn = np.meshgrid(np.arange(-K, K + 1), lags, indexing='ij')
    keep = np.abs(D) >= float(prune) * np.abs(D).max() if prune else np.ones(D.shape, dtype=bool)
    return mm[keep].astype(np.int32), nn[keep].astype(np.int32), D[keep]


def xpm_channels(xpm, ich: int, nch: int):
    """the interferers (1-based) of channel ich among nch: a list of channels, 'adjacent' (ich -+ 1 where they exist) or
    'all' (every other channel)"""
    if isinstance(xpm, str):
        if xpm == 'adjacent':
            return [c for c in (ich - 1, ich + 1) if 1 <= c <= nch]
        if xpm == 'all':
            return [c for c in range(1, nch + 1) if c != ich]
        raise ValueError("xpm must be a list of channels, 'adjacent' or 'all', got %r" % (xpm,))
    out = [int(c) for c in xpm]
    for c in out:
        if c < 1 or c > nch:
            raise ValueError('xpm: channel %d does not exist' % c)
        if c == ich:
            raise ValueError('xpm: channel %d is the compensated channel itself' % c)
    if len(set(out)) != len(out):
        raise ValueError('xpm: a channel is listed twice')
    if not out:
        raise ValueError('xpm: no interferer')
    return out


def xpm_shifts(xpm, ich: int, G=None):
    """the receiver's shifts (channel_ndfn) of the interferers xpm_channels gives"""
    from .receiver import channel_ndfn
    G = G or GSTATE
    return [int(channel_ndfn(c, G)) for c in xpm_channels(xpm, int(ich), int(G.NCH))]


def scale_factor(setup: FiberSetup, nspan: int, gain_db: Optional[float] = None) -> float:
    """s = (exp(alpha*Ls/2)/sqrt(G))^nspan (G = 1 without an amplifier): the factor that brings the received field to
    launch scale, the net of DBP's per-step and per-span factors"""
    g = 1.0 if gain_db is None else 10 ** (gain_db * 0.1)
    return (math.exp(0.5 * setup.alphalin * setup.length) / math.sqrt(g)) ** int(nspan)


def pb_plan(ctx: _lib.Context, setup: FiberSetup, nspan: int, gain_db: Optional[float] = None, xi: float = 1.0,
            K: int = 16, prune: float = 0.0, pulse=None, batch: int = 1, nt: Optional[int] = None, nquad: int = 32,
            window: Optional[int] = None, coefs=None, shift: Optional[int] = None,
            decim: Optional[int] = None, table: str = 'host', xpm=None, xpm_coefs=None) -> _lib.PbPlan:
    """The PB-NLC stage of nspan spans of the fiber `setup` describes (amplifier of gain_db [dB] after each; None: none), for
    resident one-column FP64 fields of `batch` realizations: pmx_pb_create with the table of pb_coefficients (or `coefs`,
    a (m, n, C) table), the model and gamma of the fiber, and s = scale_factor(setup, nspan, gain_db).
    decim: single-channel PB-NLC of a one-column field (pmx_pb_channel_create) -- the channel that `shift` bins bring to
    baseband (the receiver's ndfn; default 0), compensated on nfft/decim samples with the table of channel_setup at
    nt/decim samples per symbol; the pulse (and a `coefs` table) then belong to that rate, the default pulse is
    channel_pulse.  table: 'host' computes the table with numpy (pb_coefficients), 'device' with the library on ctx's device
    (pmx_pb_table); the two agree to rounding.
    xpm: XPM-aware single-channel PB-NLC (pmx_pb_xpm_create) with the interferers that these shifts bring to baseband,
    each with its table of xpm_coefficients (K, prune and nquad as for the channel's own table) or xpm_coefs[c], a (m, n,
    D) table per interferer.  A request the library refuses raises ValueError with its message, before any table is
    computed."""
    nt = int(nt or GSTATE.NT)
    _check_table(table)
    if decim is None and shift is not None:
        raise ValueError('pb_plan: shift selects a channel for single-channel PB-NLC and needs decim')
    if xpm is not None and decim is None:
        raise ValueError('pb_plan: xpm takes the interferers of single-channel PB-NLC and needs decim')
    if xpm_coefs is not None and xpm is None:
        raise ValueError('pb_plan: xpm_coefs needs xpm')
    full, nt_full = setup, nt
    if setup.nfc != 1:
        raise ValueError('pmx_pb_create: nfc=%d, PB-NLC takes one-column fields holding one channel' % setup.nfc)
    _lib.check_pb_k(K)
    band = None
    if decim is not None:
        r = _check_decim(decim, nt)
        if pulse is None:
            pulse = channel_pulse(nt, r, setup.nfft)
        band = _lib.make_band(shift or 0, r)
        setup, nt = channel_setup(setup, shift or 0, r), nt // r
    p = np.asarray(synth.cosroll_pulse(nt, 0.2) if pulse is None else pulse, dtype=np.float64).ravel()
    w, gam = model_weights(setup)
    args = (setup.nfft // nt, nt, batch, p, w, gam, xi, scale_factor(setup, nspan, gain_db))
    if xpm is not None:            # the library's checks first, on placeholder tables
        shifts = [int(v) for v in np.ravel(xpm)]
        wx, _ = xpm_weights(setup)
        one = ([0], [0], [0.0])
        _lib.check_pb_xpm(_lib.make_pb(*args, *one), band, _lib.make_pb_xpm(shifts, [one] * len(shifts), wx))
    if coefs is None:
        coefs = pb_coefficients(setup, nspan, p, K, prune, nt, nquad, window, ctx=ctx if table == 'device' else None)
    if xpm is None:
        m, n, C = coefs
        return _lib.PbPlan(ctx, _lib.make_pb(*args, m, n, C), band)
    if xpm_coefs is None:
        xpm_coefs = [xpm_coefficients(full, nspan, shift or 0, sc, r, p, K, prune=prune, nt=nt_full, nquad=nquad)
                     for sc in shifts]
    desc, xd = _lib.make_pb(*args, *coefs), _lib.make_pb_xpm(shifts, xpm_coefs, wx)
    _lib.check_pb_xpm(desc, band, xd)
    return _lib.PbPlan(ctx, desc, band, xd)


def pbnlc(x, flag: str, nspan: int = 1, gain_db: Optional[float] = None, xi: float = 1.0, K: int = 16, prune: float = 0.0,
          pulse=None, ctx: Optional[_lib.Context] = None, nquad: int = 32, window: Optional[int] = None,
          ich: Optional[int] = None, decim: Optional[int] = None, table: str = 'host', xpm=None):
    """Compensates GSTATE.FIELDX / FIELDY in place for nspan spans of the fiber x, the amplifier of gain_db [dB] after each
    (None: no amplifier): the all-pass step that undoes the link's chromatic dispersion (as Link.cd_plan), then the PB-NLC
    stage with the triplet table of K (pb_coefficients) at s = scale_factor(...), the fraction xi of the perturbation
    subtracted.  The nonlinear model is the one fiber() used: Manakov when x.manakov is 'yes' and the flag has 'p', else the
    CNLSE.  One channel (GSTATE.NCH == 1), two polarizations, FP64.  ich, decim: single-channel PB-NLC of channel ich
    (1-based) of a 'unique' multiplex of any NCH on nfft/decim samples (pb_plan; a given pulse is at that rate); afterwards
    the field holds that channel alone, on its own bins.  table: 'host' (numpy) or 'device' (pmx_pb_table) computes the
    triplet table (pb_plan).  xpm (with ich and decim): XPM-aware PB-NLC with the symbols of these channels (1-based), of
    the adjacent ones ('adjacent') or of all others ('all') (pb_plan's xpm, at their receiver shifts).  The field stays
    resident on the device like dbp() leaves it."""
    from .mc import cd_plan_of
    G = GSTATE
    _check_table(table)
    f = str(flag).lower()
    if len(f) != 4:
        raise ValueError("wrong flag. E.g. flag can be 'g---','gp--','-s--', etc")
    shift = None
    if xpm is not None and decim is None:
        raise ValueError('pbnlc: xpm takes the interferers of single-channel PB-NLC and needs ich and decim')
    if decim is not None:
        if ich is None:
            raise ValueError('pbnlc: single-channel PB-NLC (decim) needs the channel ich')
        if ich < 1 or ich > G.NCH:
            raise ValueError('The channel does not exist')
        if G.field_shape()[1] != 1:
            raise ValueError("pbnlc: single-channel PB-NLC takes a field holding every channel in one column ('unique')")
        _check_decim(decim, G.NT)
        from .receiver import channel_ndfn
        shift = int(channel_ndfn(ich, G)) if G.NCH > 1 else 0
        if xpm is not None:
            xpm = xpm_shifts(xpm, ich, G)
    elif ich is not None:
        raise ValueError('pbnlc: ich selects a channel for single-channel PB-NLC and needs decim')
    elif G.NCH != 1:
        raise ValueError('pbnlc: PB-NLC takes a field holding one channel (GSTATE.NCH == 1), got %d' % G.NCH)
    if not G.has_y():
        raise ValueError('pbnlc: PB-NLC takes two-polarization fields (FIELDY is empty)')
    if G.field_shape()[1] != 1:
        raise ValueError('pbnlc: PB-NLC takes one-column fields')
    if int(nspan) < 1:
        raise ValueError('pbnlc: nspan must be >= 1')
    _lib.check_pb_k(K)
    s = fiber_setup(x, f[0] + '-' + f[2:])
    s.manakov = f[1] == 'p' and str(_get(x, 'manakov', 'no')) == 'yes'
    ctx = ctx or _lib.default_context()
    cd = cd_plan_of(ctx, s, int(nspan), 1, precision='f64')
    try:
        plan = pb_plan(ctx, s, nspan, gain_db, xi, K, prune, pulse, nquad=nquad, window=window, shift=shift, decim=decim,
                       table=table, xpm=xpm)
    except Exception:
        cd.close()
        raise
    fld, hx, hy = G.take_device(ctx, _lib.PMX_F64)
    try:
        cd.execute(fld)
        plan.execute(fld)
    except Exception:
        fld.close()
        raise
    finally:
        plan.close()
        cd.close()
    G.put_device(fld, hx, hy)
