"""Single-channel digital backpropagation restated in numpy (TEST INFRASTRUCTURE): the oracle of pmx_dbp_channel_create.

Built on the full-field oracles without a new operator: the spectrum of the one-column field is cropped to the channel's
M = nfft/decim bins (k - shift) mod nfft, signed k in [-M/2, M/2), at baseband; the full-field oracle (tests/dbp_oracle.py,
tests/dbp_pmd_oracle.py or tests/dbp_scalar_oracle.py) runs on that M-sample field with the cropped betat / db1; the result
is zero-padded back onto the channel's bins.  tests/test_dbp_channel.py ties it to the full-field oracle (xi = 0: the full
DBP followed by the ideal band-pass) and to the forward oracle (the exact inverse of a link run on the channel alone).
FP64 only; never imported by the product package.
"""
import numpy as np

import dbp_oracle
import dbp_pmd_oracle
import dbp_scalar_oracle


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


def dbp_channel(ux, uy, betat, gam, alphalin, lf, manakov, shift, decim, db1=None, brfs=None, spm=1, **kw):
    """Two polarizations, one column ([nfft, 1] each): dbp_oracle.dbp, or with brfs dbp_pmd_oracle.dbp_pmd, of the channel
    on nfft/decim samples; schedule, xi and gain as those take them."""
    nfft = ux.shape[0]
    b = channel_bins(nfft, shift, decim)
    cx, cy = crop(ux, b, decim), crop(uy, b, decim)
    bt = np.asarray(betat, dtype=np.float64).reshape(nfft, 1)[b]
    if brfs is None:
        vx, vy = dbp_oracle.dbp(cx, cy, bt, gam, alphalin, 1, lf, manakov, spm=spm, **kw)
    else:
        d1 = np.asarray(db1, dtype=np.float64).reshape(nfft, 1)[b]
        vx, vy = dbp_pmd_oracle.dbp_pmd(cx, cy, bt, d1, gam, alphalin, 1, lf, manakov, brfs, spm=spm, **kw)
    return embed(vx, b, nfft, decim), embed(vy, b, nfft, decim)


def dbp_channel_scalar(u, betat, gam, alphalin, lf, shift, decim, spm=1, **kw):
    """The scalar path, one column ([nfft, 1]): dbp_scalar_oracle.dbp_scalar of the channel on nfft/decim samples."""
    nfft = u.shape[0]
    b = channel_bins(nfft, shift, decim)
    bt = np.asarray(betat, dtype=np.float64).reshape(nfft, 1)[b]
    v = dbp_scalar_oracle.dbp_scalar(crop(u, b, decim), bt, gam, alphalin, 1, lf, spm=spm, **kw)
    return embed(v, b, nfft, decim)
