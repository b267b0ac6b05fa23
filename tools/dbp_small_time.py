"""Times digital backpropagation of small fields (the single-launch on-chip kernel) against the forward fiber().

    python tools/dbp_small_time.py [--reps 20] [--out DIR]

In one process, for each case: the forward fiber (pmx_fiber_exec, one launch that also runs the step control) on a
resident batch, then DBP (pmx_dbp_exec) of the same batch with the forward run's own steps (its trace_dz, xi = 1).
Cases: 2^10 two-polarization Manakov 'g-s-' at batch 1, 148 and 1184; the ex10_wdm.m shape (64 x 32 samples x 5
'sepfields' columns, scalar path 'g-sx') at batch 148; 2^12 scalar 'g-s-' at batch 148.  Reported: the median wall time
of a call (it returns synchronised), us per step and GSa*steps/s = batch*nfc*nfft*steps/time.  The card's name and power
limit are printed with the numbers.
--filter-bw BW / --taps K: also filtered DBP (BW GHz; with --taps alone 4 GHz) and, with --taps, enhanced split-step DBP
with the 2K+1 taps of dbp_time.essfm_taps, with the same steps, alternated with the forward run and plain DBP."""
import argparse
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
from polmux_b200.fiber import fiber_setup, setup_to_desc  # noqa: E402
from dbp_time import essfm_taps  # noqa: E402


def card():
    try:
        q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = 'nvidia-smi unavailable (%s)' % e
    return q


def two_pol_case(nsymb, nt):
    ex, ey, _, _ = synth.pdm_qpsk(nsymb, nt, 1)
    pmx.reset_all(nsymb, nt, 1)
    G = pmx.GSTATE
    G.SYMBOLRATE, G.LAMBDA, G.POWER = 28.0, np.array([1550.0]), np.array([2.0])
    pmx.create_field('unique', ex, ey, {'power': 'average'})
    fib = dict(synth.SMF)
    fib['length'] = 8e4
    s = fiber_setup(fib, 'g-s-')
    s.manakov = True
    return s, np.ascontiguousarray(np.asarray(G.FIELDX).T)[None], np.ascontiguousarray(np.asarray(G.FIELDY).T)[None]


def scalar_case(nsymb, nt, nch, flag):
    ex, _, _, _ = synth.pdm_qpsk(nsymb, nt, nch)
    pmx.reset_all(nsymb, nt, nch)
    G = pmx.GSTATE
    G.SYMBOLRATE, G.LAMBDA, G.POWER = 10.0, synth.wdm_lambdas(nch, 1550.0, 0.4), np.full(nch, 4.0)
    pmx.create_field('sepfields' if nch > 1 else 'unique', ex, None, {'power': 'average'})
    fib = dict(synth.SMF)
    fib.update(length=1e5, dphimax=3e-3)
    s = fiber_setup(fib, flag)
    x = np.ascontiguousarray(np.asarray(G.FIELDX).T)[None]
    return s, x, np.zeros_like(x)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--filter-bw', type=float, default=None,
                    help='also filtered DBP [GHz] with the same steps, alternated with the forward run and plain DBP')
    ap.add_argument('--taps', type=int, default=None,
                    help='also enhanced split-step DBP with 2K+1 taps, alternated with the others')
    ap.add_argument('--out', default=None, help='directory for dbp_small_time.json')
    a = ap.parse_args()
    ctx = _lib.default_context(0)
    cases = [('2^10 2pol Manakov g-s-', lambda: two_pol_case(64, 16), b) for b in (1, 148, 1184)]
    cases += [('ex10 64x32x5 scalar g-sx', lambda: scalar_case(64, 32, 5, 'g-sx'), 148),
              ('2^12 scalar g-s-', lambda: scalar_case(128, 32, 1, 'g-s-'), 148)]
    rows = []
    for name, make, B in cases:
        s, x1, y1 = make()
        n, nfc = s.nfft, s.nfc
        tx = _lib.DeviceField(ctx, n, nfc, 1)
        tx.upload(x1, y1)
        fld = _lib.DeviceField(ctx, n, nfc, B)
        desc, keep = setup_to_desc(s, batch=B)
        fwd = _lib.Plan(ctx, desc, keep)
        fld.broadcast_from(tx)
        res = fwd.execute(fld, trace_cap=4096)                     # (also the warm-up of the forward kernel)
        dz, _ = res.schedule(0)
        steps = len(dz)
        dbp = dbp_plan(ctx, s, 1, None, step_len=dz, batch=B)
        fld.broadcast_from(tx)
        dbp.execute(fld)                                           # warm-up
        runs = [('forward', lambda: fwd.execute(fld)), ('dbp', lambda: dbp.execute(fld))]
        filt = ess = None
        if a.filter_bw is not None or a.taps is not None:
            filt = dbp_plan(ctx, s, 1, None, step_len=dz, batch=B, filter_bw=4.0 if a.filter_bw is None else a.filter_bw)
            fld.broadcast_from(tx)
            filt.execute(fld)                                      # warm-up
            runs.append(('filtered', lambda: filt.execute(fld)))
        if a.taps is not None:
            ess = dbp_plan(ctx, s, 1, None, step_len=dz, batch=B, nl_taps=essfm_taps(a.taps))
            fld.broadcast_from(tx)
            ess.execute(fld)                                       # warm-up
            runs.append(('essfm', lambda: ess.execute(fld)))
        t = {what: [] for what, _ in runs}
        for _ in range(a.reps):                                    # they alternate
            for what, run in runs:
                fld.broadcast_from(tx)
                ctx.sync()
                t0 = time.perf_counter()
                run()
                t[what].append(time.perf_counter() - t0)
        fwd.close()
        dbp.close()
        if filt is not None:
            filt.close()
        if ess is not None:
            ess.close()
        fld.close()
        tx.close()
        row = dict(case=name, batch=B, nfft=n, nfc=nfc, steps=steps)
        for what, v in t.items():
            med = float(np.median(v))
            row[what] = dict(seconds_median=med, spread=[float(min(v)), float(max(v))], us_per_step=med / steps * 1e6,
                             gsa_steps_per_s=B * nfc * n * steps / med / 1e9)
        row['dbp_vs_forward'] = row['dbp']['gsa_steps_per_s'] / row['forward']['gsa_steps_per_s']
        rows.append(row)
        if filt is not None:
            print('%-26s batch %5d  filtered dbp %8.2f us/step %7.2f GSa*steps/s | filtered/dbp %.3f'
                  % (name, B, row['filtered']['us_per_step'], row['filtered']['gsa_steps_per_s'],
                     row['filtered']['gsa_steps_per_s'] / row['dbp']['gsa_steps_per_s']))
        if ess is not None:
            print('%-26s batch %5d  essfm dbp %8.2f us/step %7.2f GSa*steps/s | essfm/dbp %.3f | essfm/filtered %.3f'
                  % (name, B, row['essfm']['us_per_step'], row['essfm']['gsa_steps_per_s'],
                     row['essfm']['gsa_steps_per_s'] / row['dbp']['gsa_steps_per_s'],
                     row['essfm']['gsa_steps_per_s'] / row['filtered']['gsa_steps_per_s']))
        print('%-26s batch %5d  %3d steps | forward %8.2f us/step %7.2f GSa*steps/s | dbp %8.2f us/step %7.2f GSa*steps/s'
              ' | dbp/forward %.3f' % (name, B, steps, row['forward']['us_per_step'], row['forward']['gsa_steps_per_s'],
                                       row['dbp']['us_per_step'], row['dbp']['gsa_steps_per_s'], row['dbp_vs_forward']))
    info = card()
    print('card: %s' % info)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        json.dump(dict(card=info, rows=rows), open(os.path.join(a.out, 'dbp_small_time.json'), 'w'), indent=1)


if __name__ == '__main__':
    main()
