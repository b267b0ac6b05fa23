"""Single-channel PB-NLC restated in numpy (TEST INFRASTRUCTURE): the oracle of pmx_pb_channel_create.

The stage oracle of tests/pbnlc_oracle.py on the channel's spectrum cropped to nfft/decim samples, with dbp_oracle's crop
and embed, as dbp_oracle.dbp_channel does it for DBP.  Never imported by the product package.
"""
import numpy as np

from dbp_oracle import channel_bins, crop, embed
from pbnlc_oracle import stage


def pb_channel(ux, uy, pulse, nt, m, n, C, weights, gamma, scale, xi, shift, decim):
    """single-channel PB-NLC of one realization ([nfft] each): crop to the channel's nfft/decim bins at baseband, stage at
    that rate (pulse and nt = samples per symbol there), embed back on the channel's bins -> (ux, uy, A, Delta)"""
    N = len(np.ravel(ux))
    b = channel_bins(N, shift, decim)
    vx, vy = crop(np.ravel(ux), b, decim), crop(np.ravel(uy), b, decim)
    rx, ry, A, D = stage(vx, vy, pulse, nt, m, n, C, weights, gamma, scale, xi)
    return embed(rx, b, N, decim), embed(ry, b, N, decim), A, D
