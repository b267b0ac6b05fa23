"""Perturbation-based nonlinearity compensation restated in numpy (TEST INFRASTRUCTURE): the oracle of pb_coefficients and of
pmx_pb_create / pmx_pb_exec.

The model weights come from the library's own nonlinear step (matrix_nl_step, fiber.m:827-851).  Its CNLSE step is
u <- R(phi) exp(-j*gam*leff*P) u with P = |ux|^2 + |uy|^2, s3 = 2*Im(conj(ux)*uy) and the rotation by phi = gam*leff*s3/3
(uxx = cos(phi)*ux + sin(phi)*uy, uyy = -sin(phi)*ux + cos(phi)*uy), so to first order in leff
    dux = -j*gam*P*ux + gam*(s3/3)*uy,     s3 = -j*(conj(ux)*uy - ux*conj(uy)),
    dux = -j*gam*[ |ux|^2 ux + |uy|^2 ux + (1/3)*(conj(ux)*uy^2 - |uy|^2 ux) ]
        = -j*gam*[ |ux|^2 ux + (2/3)*|uy|^2 ux + (1/3)*uy^2 conj(ux) ],
and duy with x <-> y (the sign of the rotation flips with the roles): (a, b, c) = (1, 2/3, 1/3).  The Manakov step is the
phase alone with gam*8/9: (1, 1, 0).  Expanding u = sum_i A_i g_i in pulses and keeping the triplets i + j - l = k of the
projection onto g_k gives the sum polmux_ssfm.h states.

coefficients_direct evaluates the overlap integral term by term (the forward oracle's lin_step on the whole block, every
(m, n), its own Gauss-Legendre nodes): slow, for small K, the check of the FFT form of pb_coefficients.  project, triplets and
reconstruct are the three device kernels, the triplet sum in the device's order (list order, one accumulation per entry).
Never imported by the product package.
"""
import numpy as np

import oracle.fiber_oracle as orc


def nodes(length, nspan, alphalin, nquad):
    x, w = np.polynomial.legendre.leggauss(int(nquad))
    z = 0.5 * length * (x + 1.0)
    wz = 0.5 * length * w * np.exp(-alphalin * z)
    return [(s * length + zz, ww) for s in range(int(nspan)) for zz, ww in zip(z, wz)]


def pulse_at(pulse, nt, N, k):
    """[N] the pulse of symbol k, centred at time index k*nt, circular"""
    p = np.zeros(N, dtype=np.complex128)
    p[(k * nt + np.arange(len(pulse)) - len(pulse) // 2) % N] = pulse
    return p


def coefficients_direct(betat, length, alphalin, nspan, pulse, nt, K, nquad):
    """-> C [2K+1][2K+1] (index m+K, n+K) of the overlap integral, on the whole grid of betat"""
    N = len(betat)
    bt = np.asarray(betat, dtype=np.float64).reshape(N, 1)
    norm = float(np.sum(np.asarray(pulse) ** 2))
    C = np.zeros((2 * K + 1, 2 * K + 1), dtype=np.complex128)
    base = pulse_at(pulse, nt, N, 0).reshape(N, 1)
    for z, w in nodes(length, nspan, alphalin, nquad):
        g0 = orc.lin_step(bt * z, base)[:, 0]
        g = {m: np.roll(g0, m * nt) for m in range(-2 * K, 2 * K + 1)}
        for m in range(-K, K + 1):
            for n in range(-K, K + 1):
                C[m + K, n + K] += w * np.sum(np.conj(g0) * g[m] * g[n] * np.conj(g[m + n])) / norm
    return C


def project(ux, uy, pulse, nt):
    """-> A [2][nsymb]: sum_j p[j] u[(k*nt - np/2 + j) mod N] / sum p^2"""
    N = len(ux)
    nsymb = N // nt
    idx = (np.arange(nsymb)[:, None] * nt - len(pulse) // 2 + np.arange(len(pulse))[None, :]) % N
    norm = float(np.sum(np.asarray(pulse) ** 2))
    return np.stack([(u[idx] * pulse[None, :]).sum(axis=1) / norm for u in (np.ravel(ux), np.ravel(uy))])


def fold(m, n, C, gamma, scale):
    """C' = -j*gamma*s^2*C as pmx_pb_create forms it"""
    g = gamma * scale * scale
    C = np.asarray(C, dtype=np.complex128)
    return g * C.imag - 1j * (g * C.real)


def triplets(A, m, n, C, weights, gamma, scale=1.0):
    """-> Delta [..., 2, nsymb] = sum_i C'_i T_i(k), list order (A [..., 2, nsymb]: leading axes are realizations)"""
    a, b, c = weights
    A = np.asarray(A, dtype=np.complex128)
    x, y = A[..., 0, :], A[..., 1, :]
    cf = fold(m, n, C, gamma, scale)
    D = np.zeros_like(A)
    for mi, ni, ci in zip(np.ravel(m), np.ravel(n), cf):
        xm, ym = np.roll(x, -mi, axis=-1), np.roll(y, -mi, axis=-1)
        xn, yn = np.roll(x, -ni, axis=-1), np.roll(y, -ni, axis=-1)
        xs, ys = np.roll(x, -(mi + ni), axis=-1), np.roll(y, -(mi + ni), axis=-1)
        tx = (a * xm * xn + c * ym * yn) * np.conj(xs) + b * xm * yn * np.conj(ys)
        ty = (a * ym * yn + c * xm * xn) * np.conj(ys) + b * ym * xn * np.conj(xs)
        D[..., 0, :] += ci * tx
        D[..., 1, :] += ci * ty
    return D


def reconstruct(ux, uy, D, pulse, nt, xi):
    """u[t] -= xi * sum_k Delta_k p[t - k*nt + np/2]"""
    N = len(ux)
    nsymb = N // nt
    ox, oy = np.array(np.ravel(ux), dtype=np.complex128), np.array(np.ravel(uy), dtype=np.complex128)
    sx, sy = np.zeros(N, dtype=np.complex128), np.zeros(N, dtype=np.complex128)
    for j in range(len(pulse)):                           # (for one j the samples of the symbols are distinct)
        t = (np.arange(nsymb) * nt + j - len(pulse) // 2) % N
        sx[t] += pulse[j] * D[0]
        sy[t] += pulse[j] * D[1]
    return ox - xi * sx, oy - xi * sy


def stage(ux, uy, pulse, nt, m, n, C, weights, gamma, scale, xi):
    """the whole device stage on one realization -> (ux, uy, A, Delta)"""
    A = project(ux, uy, pulse, nt)
    D = triplets(A, m, n, C, weights, gamma, scale)
    rx, ry = reconstruct(ux, uy, D, pulse, nt, xi)
    return rx, ry, A, D
