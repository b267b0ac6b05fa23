"""Times digital backpropagation (pmx_dbp_exec) against the forward link on one resident C2 batch.

    python tools/dbp_time.py [--batch 16] [--nsymb 65536] [--reps 3] [--pmd] [--out DIR]

C2 (BASELINE.md): 10 x 80 km Manakov spans, 16 dB amplifiers, 2^16 symbols x 16 samples = 2^20 samples.  In one process:
the forward link (pmx_link_exec, noise-free, 'g-s-' with the Manakov model: the nonlinear-phase step control) and DBP of
the same 10 spans with M = 1, 4 and 16 uniform steps per span.  Reported per run: wall time of the call (it returns
synchronised), GSa*steps/s = batch*nfft*steps/time and the share of the HBM roofline for the 192 algorithmic bytes a
step moves per Sa in FP64 (3 passes x read + write x 32 B), against the same peak bench.py uses (MEASURED_PEAKS.json
hbm_gbs, else 6650 GB/s).  The card's name and power limit are printed with the numbers.
--pmd: the 'gps-' C2 link with 100 plates per span and a plate draw per span and realization; timed are the forward link,
PMD-blind DBP and PMD-aware DBP (each at M = 1, 4, 16) and the genie equaliser (Link.equalize, one 100-trunk step per
span).
--taps K: enhanced split-step DBP with the 2K+1 taps of essfm_taps (symmetric, sum 1) at 1, 2 and 4 steps per span,
alternated in this process with the plain plan and the filtered plan (--filter-bw, default 4 GHz)."""
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

BYTES_PER_SA_STEP = 192.0


def essfm_taps(k):
    """the fixed symmetric test tap set of --taps K: 2K+1 samples of a Gaussian, normalised to sum 1"""
    m = np.arange(-k, k + 1, dtype=np.float64)
    c = np.exp(-(m / (0.5 * k + 1)) ** 2)
    return c / c.sum()


def card():
    try:
        q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = 'nvidia-smi unavailable (%s)' % e
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=16)
    ap.add_argument('--nsymb', type=int, default=1 << 16)
    ap.add_argument('--nt', type=int, default=16)
    ap.add_argument('--nspan', type=int, default=10)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--pmd', action='store_true', help="the 'gps-' link with 100 plates; PMD-aware DBP and the equaliser too")
    ap.add_argument('--filter-bw', type=float, default=None,
                    help='filtered DBP [GHz] at 1, 2 and 4 steps per span, alternated with the plain plan in this process')
    ap.add_argument('--taps', type=int, default=None,
                    help='enhanced split-step DBP with 2K+1 taps, alternated with plain and filtered DBP in this process')
    ap.add_argument('--out', default=None, help='directory for dbp_time.json')
    a = ap.parse_args()
    try:
        peak = float(json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json'))).get('hbm_gbs', 6650.0))
    except Exception:  # noqa: BLE001
        peak = 6650.0
    ex, ey, _, _ = synth.pdm_qpsk(a.nsymb, a.nt, 1)
    pmx.reset_all(a.nsymb, a.nt, 1)
    G = pmx.GSTATE
    G.SYMBOLRATE, G.LAMBDA, G.POWER = 28.0, np.array([1550.0]), np.array([2.0])
    pmx.create_field('unique', ex, ey, {'power': 'average'})
    fib = dict(synth.SMF)
    fib['length'] = 8e4
    if a.pmd:
        fib.update(dgd=0.3, nplates=100, manakov='yes')
        s = fiber_setup(fib, 'gps-', rng=np.random.Generator(np.random.PCG64(0)))
    else:
        s = fiber_setup(fib, 'g-s-')
    s.manakov = True
    ctx = _lib.default_context(0)
    B, n = a.batch, s.nfft
    tx = _lib.DeviceField(ctx, n, 1, 1)
    tx.upload(G.FIELDX_TX, G.FIELDY_TX)
    fld = _lib.DeviceField(ctx, n, 1, B)
    gain = 10 ** 1.6
    desc, keep = setup_to_desc(s, batch=B)
    fwd = _lib.Plan(ctx, desc, keep)
    link, lkeep = _lib.make_link(a.nspan, gain)
    rows = []

    def timed(name, run, steps_of, reps=None):
        for rep in range((a.reps if reps is None else reps) + 1):   # the first call warms up (module load, tables)
            fld.broadcast_from(tx)
            ctx.sync()
            t0 = time.perf_counter()
            out = run()
            dt = time.perf_counter() - t0
            if rep == 0:
                continue
            steps = steps_of(out)
            sa = float(steps) * n
            rows.append(dict(run=name, rep=rep, seconds=dt, steps_per_realization=steps / B,
                             gsa_steps_per_s=sa / dt / 1e9, roofline_share=BYTES_PER_SA_STEP * sa / (peak * 1e9) / dt))
            print('%-14s rep %d  %8.2f ms  %6d steps/realization  %7.2f GSa*steps/s  %5.1f %% of %.0f GB/s x 192 B'
                  % (name, rep, dt * 1e3, steps / B, rows[-1]['gsa_steps_per_s'], 100 * rows[-1]['roofline_share'], peak))

    if a.pmd:
        fwd.close()
        from polmux_b200 import mc
        lk = mc.Link(ctx, s, a.nspan, B, 16.0, None)        # noise-free, a plate draw per span and realization
        plates = tuple(np.stack([pl[i] for pl in lk.plates]) for i in range(3))
        timed('forward', lambda: lk.run(fld, 1), lambda r: r // n)
    else:
        timed('forward', lambda: fwd.link_exec(fld, link, lkeep), lambda r: int(r.ncycle.sum()))
    for m in (1, 4, 16):
        plan = dbp_plan(ctx, s, a.nspan, 16.0, steps_per_span=m, batch=B)
        timed('dbp M=%d' % m, lambda: plan.execute(fld), lambda _r, m=m: m * a.nspan * B)
        plan.close()
    if a.filter_bw is not None or a.taps is not None:
        bw = 4.0 if a.filter_bw is None else a.filter_bw
        for m in (1, 2, 4):
            plans = [('dbp M=%d' % m, dbp_plan(ctx, s, a.nspan, 16.0, steps_per_span=m, batch=B)),
                     ('filtered M=%d' % m, dbp_plan(ctx, s, a.nspan, 16.0, steps_per_span=m, batch=B, filter_bw=bw))]
            if a.taps is not None:
                plans.append(('essfm M=%d' % m, dbp_plan(ctx, s, a.nspan, 16.0, steps_per_span=m, batch=B,
                                                          nl_taps=essfm_taps(a.taps))))
            for _ in range(a.reps):
                for name, pl in plans:
                    timed(name, lambda pl=pl: pl.execute(fld), lambda _r, m=m: m * a.nspan * B, reps=1)
            for _, pl in plans:
                pl.close()
    if a.pmd:
        for m in (1, 4, 16):
            plan = dbp_plan(ctx, s, a.nspan, 16.0, steps_per_span=m, batch=B, plates=plates)
            timed('dbp_pmd M=%d' % m, lambda: plan.execute(fld), lambda _r, m=m: m * a.nspan * B)
            plan.close()
        timed('equalize', lambda: lk.equalize(fld), lambda _r: a.nspan * B)
    info = card()
    print('card: %s' % info)
    summary = {}
    for name in sorted({r['run'] for r in rows}):
        v = [r['gsa_steps_per_s'] for r in rows if r['run'] == name]
        summary[name] = dict(gsa_steps_per_s_median=float(np.median(v)), spread=[float(min(v)), float(max(v))])
    f = summary['forward']['gsa_steps_per_s_median']
    for name, v in summary.items():
        v['vs_forward'] = v['gsa_steps_per_s_median'] / f
        print('%-14s median %7.2f GSa*steps/s  (%.3f x forward)' % (name, v['gsa_steps_per_s_median'], v['vs_forward']))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        json.dump(dict(card=info, peak_gbs=peak, batch=B, nfft=n, nspan=a.nspan, pmd=a.pmd, runs=rows, summary=summary),
                  open(os.path.join(a.out, 'dbp_time.json'), 'w'), indent=1)


if __name__ == '__main__':
    main()
