"""XPM-aware single-channel PB-NLC restated in numpy (TEST INFRASTRUCTURE): the oracle of pbnlc.xpm_coefficients and of
pmx_pb_xpm_create / pmx_pb_exec.

The weights come from the library's own nonlinear step, as tests/pbnlc_oracle.py derives the SPM ones.  With the channel of
interest (COI) A and an interferer B at another frequency, u = A + B*e (e the interferer's carrier in the COI's frame), the
terms of the step's first order at the COI's frequency that are linear in A and in B*conj(B) are, from
dux = -j*gam*[ |ux|^2 ux + (2/3)*|uy|^2 ux + (1/3)*uy^2 conj(ux) ] (CNLSE),
    |ux|^2 ux            -> 2*Ax |Bx|^2
    (2/3)*|uy|^2 ux      -> (2/3)*(Ax |By|^2 + Ay Bx conj(By))
    (1/3)*uy^2 conj(ux)  -> (2/3)*Ay By conj(Bx)
so (w1, w2, w3, w4) = (2, 2/3, 2/3, 2/3) for Ax Bx conj(Bx), Ax By conj(By), Ay Bx conj(By), Ay By conj(Bx); the Manakov step
(the phase alone, -j*gam*(|ux|^2 + |uy|^2) ux) gives (2, 1, 1, 0).  first_order evaluates the step's first-order term
numerically from matrix_nl_step itself, the check of these weights on a two-tone field.

coefficients_direct evaluates D_c[m,n] = sum_q w_q sum_t conj(g_0) g_m h_n conj(h_{m+n}) / (up * sum p^2) term by term on the
whole block (slow, for small K): the check of the FFT form of xpm_coefficients.  xpm_triplets is the device's XPM sum in
its order (list order, one accumulation per entry, starting from the given Delta); pb_xpm_channel is the whole stage.
Four-wave mixing between interferers and the triplets with i + j - l != k are left out, as in the library.  Never
imported by the product package.
"""
import numpy as np

import oracle.fiber_oracle as orc
from dbp_oracle import channel_bins, crop, embed
from pbnlc_oracle import fold, nodes, project, reconstruct, triplets


def first_order(ux, uy, manakov, gam, h):
    """the first-order term of matrix_nl_step (d/dz at z = 0, no loss) on the field (ux, uy) [N]: the fourth-order central
    difference (8*(f(h) - f(-h)) - (f(2h) - f(-2h))) / (12h) -> (dux, duy)"""
    def f(dz):
        x, y = np.array(ux, dtype=np.complex128).reshape(-1, 1), np.array(uy, dtype=np.complex128).reshape(-1, 1)
        return orc.matrix_nl_step(manakov, 0.0, [gam], dz, x, y, 1, True, False)
    r = [f(s * h) for s in (1, -1, 2, -2)]
    return tuple((8 * (r[0][i] - r[1][i]) - (r[2][i] - r[3][i]))[:, 0] / (12 * h) for i in range(2))


def frame_betat(betat, shift, ref, k):
    """per metre, the dispersion of the channel at `shift` at the signed link offsets k, in the frame of the channel at ref:
    betat[(k - shift) mod N] - betat[-shift mod N] - k * (betat[(1 - ref) mod N] - betat[(-1 - ref) mod N]) / 2"""
    bt = np.asarray(betat, dtype=np.float64).ravel()
    N = bt.size
    k = np.asarray(k, dtype=np.int64)
    c0 = 0.5 * (bt[(1 - ref) % N] - bt[(-1 - ref) % N])
    return bt[(k - shift) % N] - bt[(-shift) % N] - k * c0


def coefficients_direct(betat, shift, shift_int, decim, nt, length, alphalin, nspan, pulse, K, Kn, nquad, up):
    """-> D [2K+1][2Kn+1] (index m+K, n+Kn) of the overlap integral on the whole block of the COI's M = nfft/decim grid,
    the pulse band-limited and zero-padded in frequency to up*nt/decim samples per symbol"""
    N = len(np.ravel(betat))
    M, ntm = N // decim, nt // decim
    L, ntu = up * M, up * ntm
    p0 = np.zeros(M, dtype=np.complex128)
    p0[(np.arange(len(pulse)) - len(pulse) // 2) % M] = pulse
    P = np.fft.fft(p0)
    k = np.fft.fftfreq(L, 1.0 / L).round().astype(np.int64)
    F = np.zeros(L, dtype=np.complex128)
    for j, kk in enumerate(k):
        if abs(kk) < M // 2:
            F[j] = P[kk % M]
        elif abs(kk) == M // 2:
            F[j] = 0.5 * P[M // 2]
    F *= up
    inb = np.abs(k) <= M // 2
    bg, bh = np.zeros(L), np.zeros(L)
    bg[inb] = frame_betat(betat, shift, shift, k[inb])
    bh[inb] = frame_betat(betat, shift_int, shift, k[inb])
    norm = float(np.sum(np.asarray(pulse) ** 2)) * up
    D = np.zeros((2 * K + 1, 2 * Kn + 1), dtype=np.complex128)
    for z, w in nodes(length, nspan, alphalin, nquad):
        g0 = orc.lin_step((bg * z).reshape(L, 1), np.fft.ifft(F).reshape(L, 1))[:, 0]
        h0 = orc.lin_step((bh * z).reshape(L, 1), np.fft.ifft(F).reshape(L, 1))[:, 0]
        for m in range(-K, K + 1):
            gm = np.conj(g0) * np.roll(g0, m * ntu)
            for n in range(-Kn, Kn + 1):
                D[m + K, n + Kn] += w * np.sum(gm * np.roll(h0, n * ntu) * np.conj(np.roll(h0, (m + n) * ntu))) / norm
    return D


def xpm_triplets(A, B, m, n, D, weights, gamma, scale=1.0, delta=None):
    """-> delta + sum_i D'_i T_i(k) in list order (A, B [..., 2, nsymb]: leading axes are realizations), D' = -j*gamma*s^2*D"""
    w1, w2, w3, w4 = weights
    A, B = np.asarray(A, dtype=np.complex128), np.asarray(B, dtype=np.complex128)
    out = np.zeros_like(A) if delta is None else np.array(delta, dtype=np.complex128)
    ax, ay, bx, by = A[..., 0, :], A[..., 1, :], B[..., 0, :], B[..., 1, :]
    for mi, ni, ci in zip(np.ravel(m), np.ravel(n), fold(m, n, D, gamma, scale)):
        xm, ym = np.roll(ax, -mi, axis=-1), np.roll(ay, -mi, axis=-1)
        xn, yn = np.roll(bx, -ni, axis=-1), np.roll(by, -ni, axis=-1)
        xs, ys = np.roll(bx, -(mi + ni), axis=-1), np.roll(by, -(mi + ni), axis=-1)
        P, Q, R, S = xn * np.conj(xs), yn * np.conj(ys), xn * np.conj(ys), yn * np.conj(xs)
        out[..., 0, :] += ci * (xm * (w1 * P + w2 * Q) + ym * (w3 * R + w4 * S))
        out[..., 1, :] += ci * (ym * (w1 * Q + w2 * P) + xm * (w3 * S + w4 * R))
    return out


def channel_symbols(ux, uy, pulse, nt, shift, decim):
    """the projected symbols [2][nsymb] of the channel `shift` brings to baseband: crop, project at nt (the channel's rate)"""
    N = len(np.ravel(ux))
    b = channel_bins(N, shift, decim)
    return project(crop(np.ravel(ux), b, decim), crop(np.ravel(uy), b, decim), pulse, nt)


def pb_xpm_channel(ux, uy, pulse, nt, spm, weights, xweights, gamma, scale, xi, shift, decim, xpm):
    """XPM-aware single-channel PB-NLC of one realization ([nfft] each): spm = (m, n, C) the channel's table, xpm a list of
    (shift_c, (m, n, D)) in the device's order.  Crop the channel and every interferer, project them, the SPM triplets,
    then the XPM triplets of each interferer in turn, apply, embed -> (ux, uy, A, [B_c], Delta)"""
    N = len(np.ravel(ux))
    b = channel_bins(N, shift, decim)
    vx, vy = crop(np.ravel(ux), b, decim), crop(np.ravel(uy), b, decim)
    Bs = [channel_symbols(ux, uy, pulse, nt, sc, decim) for sc, _ in xpm]
    A = project(vx, vy, pulse, nt)
    D = triplets(A, *spm, weights, gamma, scale)
    for B, (_, tab) in zip(Bs, xpm):
        D = xpm_triplets(A, B, *tab, xweights, gamma, scale, D)
    rx, ry = reconstruct(vx, vy, D, pulse, nt, xi)
    return embed(rx, b, N, decim), embed(ry, b, N, decim), A, Bs, D
