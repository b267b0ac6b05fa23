"""Times perturbation-based nonlinearity compensation (pmx_pb_create / pmx_pb_exec) on the C2 shape, or with --decim
single-channel PB-NLC (pmx_pb_channel_create) on the C4 and C2 shapes.

    python tools/pbnlc_time.py [--nspan 10] [--reps 20] [--ks 4,8,16,32,64] [--out DIR]
    python tools/pbnlc_time.py --decim 16,32,64 [--nch 9] [--reps 5] [--out DIR]
    python tools/pbnlc_time.py --table [--nch 9] [--reps 3] [--out DIR]
    python tools/pbnlc_time.py --xpm [--nch 9] [--reps 5] [--out DIR]

C2 (BASELINE.md): one 28-GBaud PDM-QPSK channel, 2^16 symbols x 16 samples = 2^20 samples, 80 km spans with 16 dB
amplifiers, Manakov.  In one process:
  1. the triplet kernel (pmx_k_pb_triplet) alone against the coefficient count (full tables of K in --ks, (2K+1)^2 entries)
     at batch 1 and 16: its device time from torch.profiler over --reps executions, and its FP64 rate -- 52 FP64
     instructions (32 DFMA, 20 DMUL) per entry and symbol, counted from the code -- as a share of the FP64 pipe rate
     tools/ubench/fp64_rate.cu measures in the same call (its best DFMA/clk/SM x 148 SMs x the card's maximum SM clock);
  2. per group of 16 realizations: the CD all-pass step + PB-NLC (K = 32, the table of the link) against DBP at one step per
     span on the whole field (single-channel DBP of the one channel, decim 2) and full DBP, each the median wall time of
     a call that ends synchronised (the PB-NLC plan with xi = 1e-9, so that the repeated runs on one field stay bounded).
The card's name, power limit and maximum SM clock are read in the same run and printed with the numbers.

With --decim: C4 (BASELINE.md: --nch 28-GBaud channels at 50 GHz in one 'unique' field of 2^16 symbols x 64 samples =
2^22 samples, 20 x 80 km Manakov spans with 16 dB amplifiers, 1 mW per channel, one realization) and C2 (one channel,
2^16 x 16 = 2^20 samples, 10 spans, batch 16).  For every decim r of the list that divides the shape's samples per
symbol, the centre channel: the CD all-pass step + single-channel PB-NLC (xi = 1, the channel's tables of K = 16 and 32
at nt/r samples per symbol) and single-channel DBP at 1 and 4 steps per span.  All plans are made first and then run in
turn, round after round, so that they are alternated in one process; each is reported as the median over --reps rounds of
the wall time of one call on a field refreshed from the Tx (a call returns synchronised), in ms per link (per group of
the batch).  The card's name, power limit and SM clocks are read in the same run.

With --table: the triplet table on the host (pb_coefficients, numpy) against the device (pmx_pb_table) for C2 (10 spans,
nquad 32, default window) at K = 16, 32 and 64, and for the centre channel of C4 at decim 16 (channel_setup /
channel_pulse, 20 spans, K = 16).  The two are alternated in one process, round after round, after a first device call
that warms up; each is the median wall time over --reps rounds of a call that returns the table on the host.  The
device's lag sums are (K+1)^2 * Ws * nodes complex multiply-adds (Ws the window in samples), 4 DFMA each; their rate is
printed as a share of the FP64 pipe tools/ubench/fp64_rate.cu measures in the same call.  The tables are compared.

With --xpm: XPM-aware single-channel PB-NLC (pmx_pb_xpm_create) of the centre channel of C4 at decim 16 and K = 16, with
the 2 adjacent and with all 8 other channels as interferers (their tables from xpm_coefficients, default Kn -- capped at
PMX_PB_XPM_MAX_N -- pruned at 1e-4 of the largest entry; nquad 2: the timing depends on the entry count only).  In one
process: (1) the XPM kernel (pmx_k_pb_xpm) alone: its device time from torch.profiler over --reps executions and its FP64
rate -- 56 FP64 instructions (36 DFMA, 20 DMUL) per entry and symbol, counted from the code -- as a share of the FP64 pipe
fp64_rate.cu measures in the same call; (2) per link, alternated round after round as with --decim: CD + XPM-aware PB-NLC
(2 and 8 interferers), CD + single-channel PB-NLC, single-channel DBP and full-field DBP at one step per span.  The
extraction of the interferers (copy, band filter at N, gather, projection) is the XPM plan's time less the single-channel
plan's and the XPM kernel's."""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import polmux_b200 as pmx  # noqa: E402
from polmux_b200 import _lib, mc, synth  # noqa: E402
from polmux_b200.dbp import dbp_plan  # noqa: E402
from polmux_b200.fiber import fiber_setup  # noqa: E402
from polmux_b200.pbnlc import channel_pulse, channel_setup, pb_coefficients, pb_plan, pb_table, model_weights  # noqa: E402
from polmux_b200.receiver import channel_ndfn  # noqa: E402

FP64_INSTR = 52
XPM_FP64_INSTR = 56


def card():
    try:
        return subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.sm,clocks.max.sm',
                               '--format=csv,noheader'], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return 'nvidia-smi unavailable (%s)' % e


def fp64_pipe():
    """best DFMA/clk/SM of tools/ubench/fp64_rate.cu, built into a temporary directory"""
    with tempfile.TemporaryDirectory() as d:
        exe = os.path.join(d, 'fp64_rate')
        subprocess.run(['nvcc', '-arch=sm_100a', '-O3', os.path.join(ROOT, 'tools', 'ubench', 'fp64_rate.cu'), '-o', exe],
                       check=True)
        out = subprocess.run([exe], capture_output=True, text=True, check=True).stdout
    return max(float(v) for v in re.findall(r'-> ([0-9.]+) DFMA/clk/SM', out))


def kernel_ms(fn, reps, name):
    """device time of kernel `name` per call of fn, from torch.profiler"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    tot = sum(e.device_time_total for e in prof.key_averages() if name in e.key)
    return tot / reps / 1000.0


def wall_ms(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t)
    return 1000.0 * float(np.median(ts))


def channel_shape(name, nsymb, nt, nch, nspan, batch, decims, reps):
    """the rows of one shape: CD + single-channel PB-NLC (K 16, 32) and single-channel DBP (1, 4 steps/span) per decim"""
    ex, ey, _, _ = synth.pdm_qpsk(nsymb, nt, nch)
    pmx.reset_all(nsymb, nt, nch)
    G = pmx.GSTATE
    G.SYMBOLRATE, G.LAMBDA, G.POWER = 28.0, synth.wdm_lambdas(nch, 1550.0, 0.4), np.full(nch, 1.0)
    pmx.create_field('unique', ex, ey, {'power': 'average'})
    fib = dict(synth.SMF)
    fib.update(length=8e4, manakov='yes')
    s = fiber_setup(fib, 'g-s-')
    s.manakov = True
    shift = int(channel_ndfn((nch + 1) // 2)) if nch > 1 else 0
    ctx = _lib.default_context(0)
    N = s.nfft
    tx = _lib.DeviceField(ctx, N, 1, 1)
    tx.upload(G.FIELDX_TX, G.FIELDY_TX)
    fld = _lib.DeviceField(ctx, N, 1, batch)
    cd = mc.cd_plan_of(ctx, s, nspan, batch, precision='f64')
    runs = []                                            # (info, callable on fld)
    for r in decims:
        if nt % r:
            print('%s: decim %d does not divide nt = %d, skipped' % (name, r, nt))
            continue
        t0 = time.perf_counter()
        p = channel_pulse(nt, r, N)
        m, n, C = pb_coefficients(channel_setup(s, shift, r), nspan, p, 32, nt=nt // r)
        print('%s r=%d: channel table of K = 32 (%d x 80 km) in %.1f s on one host thread'
              % (name, r, nspan, time.perf_counter() - t0))
        for K in (16, 32):
            sel = (np.abs(m) <= K) & (np.abs(n) <= K)
            pb = pb_plan(ctx, s, nspan, 16.0, K=K, batch=batch, nt=nt, coefs=(m[sel], n[sel], C[sel]), shift=shift,
                         decim=r)
            runs.append((dict(run='cd+pbnlc', decim=r, K=K, ncoef=int(sel.sum())),
                         lambda f, pb=pb: (cd.execute(f), pb.execute(f), ctx.sync()), pb))
        for k in (1, 4):
            plan = dbp_plan(ctx, s, nspan, 16.0, steps_per_span=k, batch=batch, precision='f64', shift=shift, decim=r)
            runs.append((dict(run='dbp', decim=r, steps_per_span=k), lambda f, plan=plan: (plan.execute(f), ctx.sync()),
                         plan))
    times = [[] for _ in runs]
    for rep in range(reps + 1):                          # round 0 warms every plan up
        for i, (_, fn, _) in enumerate(runs):
            fld.broadcast_from(tx)
            ctx.sync()
            t0 = time.perf_counter()
            fn(fld)
            if rep:
                times[i].append(time.perf_counter() - t0)
    rows = []
    for (info, _, plan), t in zip(runs, times):
        plan.close()
        row = dict(shape=name, nfft=N, batch=batch, nspan=nspan, shift=shift, ms_per_link=1e3 * float(np.median(t)),
                   spread_ms=[1e3 * min(t), 1e3 * max(t)], **info)
        rows.append(row)
        what = ('CD + PB-NLC K=%-2d' % info['K']) if info['run'] == 'cd+pbnlc' else ('DBP %d step/span ' % info['steps_per_span'])
        print('%s batch %2d r=%-2d (2^%d)  %s %9.2f ms per link  [%.2f .. %.2f]'
              % (name, batch, info['decim'], (N // info['decim']).bit_length() - 1, what, row['ms_per_link'], *row['spread_ms']))
    cd.close()
    fld.close()
    tx.close()
    return rows


def channel_main(a):
    decims = [int(v) for v in a.decim.split(',')]
    info = card()
    print('card:', info)
    rows = channel_shape('C4', 1 << 16, 64, a.nch, 20, 1, decims, a.reps)
    rows += channel_shape('C2', 1 << 16, 16, 1, 10, 16, decims, a.reps)
    print('card (after the runs):', card())
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, 'pbnlc_channel_time.json'), 'w') as f:
            json.dump(dict(card=info, runs=rows), f, indent=1)


def table_main(a):
    import torch
    torch.cuda.init()
    info = card()
    print('card:', info)
    dfma = fp64_pipe()
    mhz = float(re.findall(r'([0-9.]+) MHz', info)[-1]) if 'MHz' in info else float('nan')
    pipe = dfma * 148 * mhz * 1e6
    print('FP64 pipe: %.1f DFMA/clk/SM (fp64_rate.cu) x 148 SMs x %.0f MHz = %.3g DFMA/s' % (dfma, mhz, pipe))
    ctx = _lib.default_context(0)
    cases = []                                           # (name, setup, nspan, pulse, K, nt)
    for name, nsymb, nt, nch, nspan, decim in (('C2', 1 << 16, 16, 1, 10, None), ('C4', 1 << 16, 64, a.nch, 20, 16)):
        ex, ey, _, _ = synth.pdm_qpsk(nsymb, nt, nch)
        pmx.reset_all(nsymb, nt, nch)
        G = pmx.GSTATE
        G.SYMBOLRATE, G.LAMBDA, G.POWER = 28.0, synth.wdm_lambdas(nch, 1550.0, 0.4), np.full(nch, 1.0)
        pmx.create_field('unique', ex, ey, {'power': 'average'})
        fib = dict(synth.SMF)
        fib.update(length=8e4, manakov='yes')
        s = fiber_setup(fib, 'g-s-')
        s.manakov = True
        if decim is None:
            for K in (16, 32, 64):
                cases.append(('%s K=%d' % (name, K), s, nspan, synth.cosroll_pulse(nt, 0.2), K, nt))
        else:
            shift = int(channel_ndfn((nch + 1) // 2)) if nch > 1 else 0
            cases.append(('%s r=%d K=16' % (name, decim), channel_setup(s, shift, decim), nspan,
                          channel_pulse(nt, decim, s.nfft), 16, nt // decim))
    rows = []
    for name, s, nspan, p, K, nt in cases:
        _, _, _, W = pb_table(ctx, s, nspan, p, K, nt=nt)                 # warm-up; the window it takes
        th, td = [], []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            host = pb_coefficients(s, nspan, p, K, nt=nt)
            th.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            dev = pb_table(ctx, s, nspan, p, K, nt=nt)
            td.append(time.perf_counter() - t0)
        c00 = abs(host[2][host[2].size // 2])
        err = float(np.abs(dev[2] - host[2]).max() / c00) if np.array_equal(dev[0], host[0]) else float('inf')
        nodes, Ws = nspan * 32, W * nt
        macs = (K + 1) ** 2 * Ws * nodes
        dms = 1e3 * float(np.median(td))
        row = dict(case=name, nfft=s.nfft, nt=nt, nspan=nspan, K=K, window=W, window_samples=Ws, nodes=nodes,
                   host_s=float(np.median(th)), device_ms=dms, device_spread_ms=[1e3 * min(td), 1e3 * max(td)],
                   lag_macs=macs, dfma_share=4 * macs / (dms * 1e-3) / pipe, max_dC_rel=err)
        rows.append(row)
        print('%-12s window %5d symbols (%6d samples), %3d nodes: host %6.2f s, device %8.2f ms [%.2f .. %.2f], '
              'lag sums at %.1f %% of the FP64 pipe, max |dC|/|C00| %.1e'
              % (name, W, Ws, nodes, row['host_s'], dms, *row['device_spread_ms'], 100 * row['dfma_share'], err))
    print('card (after the runs):', card())
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, 'pbnlc_table_time.json'), 'w') as f:
            json.dump(dict(card=info, dfma_per_clk_sm=dfma, runs=rows), f, indent=1)


def xpm_main(a):
    import torch
    from polmux_b200.pbnlc import xpm_coefficients, xpm_channels
    torch.cuda.init()
    info = card()
    print('card:', info)
    dfma = fp64_pipe()
    mhz = float(re.findall(r'([0-9.]+) MHz', info)[-1]) if 'MHz' in info else float('nan')
    pipe = dfma * 148 * mhz * 1e6
    print('FP64 pipe: %.1f DFMA/clk/SM (fp64_rate.cu) x 148 SMs x %.0f MHz = %.3g FP64 instr/s' % (dfma, mhz, pipe))
    nsymb, nt, nch, nspan, r, K = 1 << 16, 64, a.nch, 20, 16, 16
    ex, ey, _, _ = synth.pdm_qpsk(nsymb, nt, nch)
    pmx.reset_all(nsymb, nt, nch)
    G = pmx.GSTATE
    G.SYMBOLRATE, G.LAMBDA, G.POWER = 28.0, synth.wdm_lambdas(nch, 1550.0, 0.4), np.full(nch, 1.0)
    pmx.create_field('unique', ex, ey, {'power': 'average'})
    fib = dict(synth.SMF)
    fib.update(length=8e4, manakov='yes')
    s = fiber_setup(fib, 'g-s-')
    s.manakov = True
    ich = (nch + 1) // 2
    shift = int(channel_ndfn(ich))
    ctx = _lib.default_context(0)
    N = s.nfft
    p = channel_pulse(nt, r, N)
    t0 = time.perf_counter()
    spm = pb_coefficients(channel_setup(s, shift, r), nspan, p, K, nt=nt // r)
    tabs = {}
    for c in xpm_channels('all', ich, nch):
        tabs[c] = xpm_coefficients(s, nspan, shift, int(channel_ndfn(c)), r, p, K, prune=1e-4, nt=nt, nquad=2)
    print('C4 r=%d: tables in %.1f s on one host thread; XPM entries per interferer %s'
          % (r, time.perf_counter() - t0, {c: len(t[2]) for c, t in tabs.items()}))
    tx = _lib.DeviceField(ctx, N, 1, 1)
    tx.upload(G.FIELDX_TX, G.FIELDY_TX)
    fld = _lib.DeviceField(ctx, N, 1, 1)
    cd = mc.cd_plan_of(ctx, s, nspan, 1, precision='f64')
    res = {'card': info, 'dfma_per_clk_sm': dfma, 'kernel': [], 'runs': []}
    runs = []
    for name, chans in (('2 adjacent', xpm_channels('adjacent', ich, nch)), ('all %d' % (nch - 1), list(tabs))):
        pb = pb_plan(ctx, s, nspan, 16.0, K=K, nt=nt, coefs=spm, shift=shift, decim=r,
                     xpm=[int(channel_ndfn(c)) for c in chans], xpm_coefs=[tabs[c] for c in chans])
        ncoef = sum(len(tabs[c][2]) for c in chans)
        fld.broadcast_from(tx)
        ms = kernel_ms(lambda: (pb.execute(fld), ctx.sync()), a.reps, 'pmx_k_pb_xpm')
        rate = XPM_FP64_INSTR * ncoef * nsymb / (ms * 1e-3)
        row = dict(interferers=len(chans), ncoef=ncoef, xpm_kernel_ms=ms, fp64_instr_per_s=rate, pipe_share=rate / pipe)
        res['kernel'].append(row)
        print('XPM kernel, %s interferers, %6d entries: %8.3f ms  %.3g FP64 instr/s  %.1f %% of the pipe'
              % (name, ncoef, ms, rate, 100 * rate / pipe))
        runs.append((dict(run='cd+pbnlc_xpm', interferers=len(chans), ncoef=ncoef),
                     lambda f, pb=pb: (cd.execute(f), pb.execute(f), ctx.sync()), pb))
    pb = pb_plan(ctx, s, nspan, 16.0, K=K, nt=nt, coefs=spm, shift=shift, decim=r)
    runs.append((dict(run='cd+pbnlc', ncoef=len(spm[2])), lambda f, pb=pb: (cd.execute(f), pb.execute(f), ctx.sync()), pb))
    for name, kw in (('dbp_channel', dict(shift=shift, decim=r)), ('dbp_full', {})):
        plan = dbp_plan(ctx, s, nspan, 16.0, steps_per_span=1, batch=1, precision='f64', **kw)
        runs.append((dict(run=name, steps_per_span=1), lambda f, plan=plan: (plan.execute(f), ctx.sync()), plan))
    times = [[] for _ in runs]
    for rep in range(a.reps + 1):                        # round 0 warms every plan up
        for i, (_, fn, _) in enumerate(runs):
            fld.broadcast_from(tx)
            ctx.sync()
            t0 = time.perf_counter()
            fn(fld)
            if rep:
                times[i].append(time.perf_counter() - t0)
    for (info_run, _, plan), t in zip(runs, times):
        plan.close()
        row = dict(ms_per_link=1e3 * float(np.median(t)), spread_ms=[1e3 * min(t), 1e3 * max(t)], **info_run)
        res['runs'].append(row)
        print('C4 r=%d K=%d %-28s %9.2f ms per link  [%.2f .. %.2f]'
              % (r, K, json.dumps(info_run), row['ms_per_link'], *row['spread_ms']))
    single = next(x['ms_per_link'] for x in res['runs'] if x['run'] == 'cd+pbnlc')
    for x, k in zip(res['runs'][:2], res['kernel']):
        ext = (x['ms_per_link'] - single - k['xpm_kernel_ms']) / x['interferers']
        x['extraction_ms_per_interferer'] = ext
        print('extraction (copy, band filter at N, gather, projection): %.2f ms per interferer (%d interferers)'
              % (ext, x['interferers']))
    cd.close()
    fld.close()
    tx.close()
    res['card_after'] = card()
    print('card (after the runs):', res['card_after'])
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, 'pbnlc_xpm_time.json'), 'w') as f:
            json.dump(res, f, indent=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--nsymb', type=int, default=1 << 16)
    ap.add_argument('--nt', type=int, default=16)
    ap.add_argument('--nspan', type=int, default=10)
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--ks', default='4,8,16,32,64')
    ap.add_argument('--decim', default=None, help='single-channel PB-NLC at these decimations (comma list) on C4 and C2')
    ap.add_argument('--table', action='store_true', help='the triplet table on the host against the device')
    ap.add_argument('--xpm', action='store_true', help='XPM-aware single-channel PB-NLC on C4 (2 and all interferers)')
    ap.add_argument('--nch', type=int, default=9, help='channels of the C4 multiplex (with --decim, --table or --xpm)')
    ap.add_argument('--out', default=None, help='directory for pbnlc_time.json (pbnlc_channel_time.json with --decim)')
    a = ap.parse_args()
    if a.decim:
        return channel_main(a)
    if a.table:
        return table_main(a)
    if a.xpm:
        return xpm_main(a)
    import torch
    torch.cuda.init()
    info = card()
    print('card:', info)
    dfma = fp64_pipe()
    mhz = float(re.findall(r'([0-9.]+) MHz', info)[-1]) if 'MHz' in info else float('nan')
    pipe = dfma * 148 * mhz * 1e6                                   # DFMA instructions per second
    print('FP64 pipe: %.1f DFMA/clk/SM (fp64_rate.cu) x 148 SMs x %.0f MHz = %.3g FP64 instr/s' % (dfma, mhz, pipe))
    ex, ey, _, _ = synth.pdm_qpsk(a.nsymb, a.nt, 1)
    pmx.reset_all(a.nsymb, a.nt, 1)
    G = pmx.GSTATE
    G.SYMBOLRATE, G.LAMBDA, G.POWER = 28.0, np.array([1550.0]), np.array([1.0])
    pmx.create_field('unique', ex, ey, {'power': 'average'})
    fib = dict(synth.SMF)
    fib.update(length=8e4, manakov='yes')
    s = fiber_setup(fib, 'g-s-')
    s.manakov = True
    ctx = _lib.Context(0)
    N = a.nsymb * a.nt
    res = {'card': info, 'dfma_per_clk_sm': dfma, 'triplet': [], 'chain': {}}
    t0 = time.perf_counter()
    m, n, C = pb_coefficients(s, a.nspan, None, 64, nt=a.nt)
    res['table_s_K64'] = time.perf_counter() - t0
    print('table of %d x 80 km, K = 64: %.1f s on one host thread' % (a.nspan, res['table_s_K64']))
    w, gam = model_weights(s)
    p = synth.cosroll_pulse(a.nt, 0.2)
    for batch in (1, 16):
        fld = _lib.DeviceField(ctx, N, 1, batch)
        x = np.broadcast_to(np.asarray(G.FIELDX).T[None], (batch, 1, N))
        y = np.broadcast_to(np.asarray(G.FIELDY).T[None], (batch, 1, N))
        fld.upload(x, y)
        for K in [int(k) for k in a.ks.split(',')]:
            sel = (np.abs(m) <= K) & (np.abs(n) <= K)
            plan = _lib.PbPlan(ctx, _lib.make_pb(a.nsymb, a.nt, batch, p, w, gam, 1e-9, 1.0, m[sel], n[sel], C[sel]))
            ms = kernel_ms(lambda: (plan.execute(fld), ctx.sync()), a.reps, 'pmx_k_pb_triplet')
            plan.close()
            ncoef = int(sel.sum())
            rate = FP64_INSTR * ncoef * a.nsymb * batch / (ms * 1e-3)
            row = dict(batch=batch, K=K, ncoef=ncoef, triplet_ms=ms, fp64_instr_per_s=rate, pipe_share=rate / pipe)
            res['triplet'].append(row)
            print('triplet batch %2d K %2d ncoef %5d: %8.3f ms  %.3g FP64 instr/s  %.1f %% of the pipe'
                  % (batch, K, ncoef, ms, rate, 100 * rate / pipe))
        fld.close()
    # per group of 16: CD + PB-NLC against DBP at one step per span
    batch = 16
    fld = _lib.DeviceField(ctx, N, 1, batch)
    x = np.broadcast_to(np.asarray(G.FIELDX).T[None], (batch, 1, N))
    y = np.broadcast_to(np.asarray(G.FIELDY).T[None], (batch, 1, N))
    fld.upload(x, y)
    cd = mc.cd_plan_of(ctx, s, a.nspan, batch, precision='f64')
    sel = (np.abs(m) <= 32) & (np.abs(n) <= 32)
    # (xi = 1e-9: the chain runs over and over on one field, which a full correction each time would drive to overflow;
    # every xi != 0 costs the same launches and work)
    pb = pb_plan(ctx, s, a.nspan, 16.0, xi=1e-9, batch=batch, nt=a.nt, coefs=(m[sel], n[sel], C[sel]))
    res['chain']['cd_pbnlc_K32_ms'] = wall_ms(lambda: (cd.execute(fld), pb.execute(fld), ctx.sync()), a.reps)
    res['chain']['cd_ms'] = wall_ms(lambda: (cd.execute(fld), ctx.sync()), a.reps)
    for name, kw in (('dbp_channel_1step_ms', dict(decim=2, shift=0)), ('dbp_full_1step_ms', {})):
        plan = dbp_plan(ctx, s, a.nspan, 16.0, steps_per_span=1, batch=batch, precision='f64', **kw)
        res['chain'][name] = wall_ms(lambda: (plan.execute(fld), ctx.sync()), a.reps)
        plan.close()
    print('per group of 16 at 2^20, %d spans: %s' % (a.nspan, json.dumps({k: round(v, 3) for k, v in res['chain'].items()})))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, 'pbnlc_time.json'), 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
