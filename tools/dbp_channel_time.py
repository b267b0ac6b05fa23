"""Times single-channel DBP (pmx_dbp_channel_create) against full-field DBP on the C4 shape.

    python tools/dbp_channel_time.py [--nspan 20] [--batch 1] [--reps 5] [--ich 5] [--out DIR]

C4 (BASELINE.md): nine 28-GBaud channels at 50 GHz in one 'unique' field of 2^16 symbols x 64 samples = 2^22 samples,
20 x 80 km Manakov spans with 16 dB amplifiers, 1 mW per channel.  In one process, on one resident batch: full-field DBP
of the link and single-channel DBP of channel ich (default the centre one) at decim r = 16, 32 and 64, each at 1, 4 and 16
uniform steps per span.  Reported per run: ms per link (the median wall time of a call, which returns synchronised) and,
for single-channel DBP, the share spent resampling -- the band filter, decimation and interpolation at 2^22 -- taken as
1 - t(M-sample DBP alone) / t(single-channel DBP), where the M-sample DBP alone is the same plan the single-channel plan
runs inside (vector tables cropped to the channel), timed on a field of M samples.  The card's name and power limit are
read in the same run and printed with the numbers."""
import argparse
import dataclasses
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import polmux_b200 as pmx  # noqa: E402
from polmux_b200 import _lib, synth  # noqa: E402
from polmux_b200.dbp import dbp_plan  # noqa: E402
from polmux_b200.fiber import fiber_setup  # noqa: E402
from polmux_b200.receiver import channel_ndfn  # noqa: E402


def card():
    try:
        q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = 'nvidia-smi unavailable (%s)' % e
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--nsymb', type=int, default=1 << 16)
    ap.add_argument('--nt', type=int, default=64)
    ap.add_argument('--nspan', type=int, default=20)
    ap.add_argument('--batch', type=int, default=1)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--ich', type=int, default=5, help='channel of the nine (5: the centre one)')
    ap.add_argument('--decims', default='16,32,64')
    ap.add_argument('--steps', default='1,4,16')
    ap.add_argument('--out', default=None, help='directory for dbp_channel_time.json')
    a = ap.parse_args()
    nch = 9
    ex, ey, _, _ = synth.pdm_qpsk(a.nsymb, a.nt, nch)
    pmx.reset_all(a.nsymb, a.nt, nch)
    G = pmx.GSTATE
    G.SYMBOLRATE, G.LAMBDA, G.POWER = 28.0, synth.wdm_lambdas(nch, 1550.0, 0.4), np.full(nch, 1.0)
    pmx.create_field('unique', ex, ey, {'power': 'average'})
    fib = dict(synth.SMF)
    fib['length'] = 8e4
    s = fiber_setup(fib, 'g-s-')
    s.manakov = True
    m = int(channel_ndfn(a.ich))
    ctx = _lib.default_context(0)
    B, n = a.batch, s.nfft
    tx = _lib.DeviceField(ctx, n, 1, 1)
    tx.upload(G.FIELDX_TX, G.FIELDY_TX)
    fld = _lib.DeviceField(ctx, n, 1, B)
    decims = [int(v) for v in a.decims.split(',')]
    steps = [int(v) for v in a.steps.split(',')]
    rows = []

    def timed(name, plan, field, src, **info):
        t = []
        for rep in range(a.reps + 1):              # the first call warms up (module load, tables)
            field.broadcast_from(src)
            ctx.sync()
            t0 = time.perf_counter()
            plan.execute(field)
            t.append(time.perf_counter() - t0)
        ms = 1e3 * float(np.median(t[1:]))
        rows.append(dict(run=name, ms_per_link=ms, spread_ms=[1e3 * min(t[1:]), 1e3 * max(t[1:])], **info))
        return ms

    for k in steps:
        plan = dbp_plan(ctx, s, a.nspan, 16.0, steps_per_span=k, batch=B)
        full = timed('full', plan, fld, tx, steps_per_span=k)
        plan.close()
        print('steps/span %2d  full-field DBP (2^%d)       %9.2f ms per link' % (k, n.bit_length() - 1, full))
        for r in decims:
            M = n // r
            plan = dbp_plan(ctx, s, a.nspan, 16.0, steps_per_span=k, batch=B, shift=m, decim=r)
            ch = timed('channel', plan, fld, tx, steps_per_span=k, decim=r)
            plan.close()
            # the M-sample DBP alone: the channel's dispersion cropped as pmx_dbp_channel_create crops it
            kk = np.fft.fftfreq(M, 1.0 / M).round().astype(np.int64)
            sm = dataclasses.replace(s, nfft=M, betat=np.ascontiguousarray(s.betat[(kk - m) % n]),
                                     db1=np.zeros((M, 1)))
            src = _lib.DeviceField(ctx, M, 1, 1)
            src.upload(np.ascontiguousarray(G.FIELDX_TX[:: r]), np.ascontiguousarray(G.FIELDY_TX[:: r]))
            wf = _lib.DeviceField(ctx, M, 1, B)
            plan = dbp_plan(ctx, sm, a.nspan, 16.0, steps_per_span=k, batch=B, disp_mode='vector')
            inner = timed('inner', plan, wf, src, steps_per_span=k, decim=r)
            plan.close()
            wf.close()
            src.close()
            share = 1.0 - inner / ch
            rows[-2]['resample_share'] = share
            print('steps/span %2d  single-channel r=%-2d (2^%d)  %9.2f ms per link  (%.2f x full-field; down + up %.1f %%, '
                  'the M-sample DBP alone %.2f ms)' % (k, r, M.bit_length() - 1, ch, ch / full, 100 * share, inner))
    info = card()
    print('card: %s' % info)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        json.dump(dict(card=info, batch=B, nfft=n, nspan=a.nspan, ich=a.ich, shift=m, runs=rows),
                  open(os.path.join(a.out, 'dbp_channel_time.json'), 'w'), indent=1)


if __name__ == '__main__':
    main()
