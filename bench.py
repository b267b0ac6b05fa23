#!/usr/bin/env python
"""bench.py -- SSFM GSa*steps/s on B200 (BASELINE.json metric), one JSON line on rank 0.

Workload (config.workload = "C2"): PDM-QPSK, 2^16 symbols x 16 samples = 2^20 samples per
polarization, 10 spans of (80 km SMF, 'gps-' Manakov, 100 random waveplates, DGD 0.1 symbol)
each followed by a 16 dB flat amplifier with ASE (noise figure 5 dB), FP64.  One "step" is
one pass of that 10-span link over a batch of independent realizations (different plate
draws and ASE seeds, same Tx field) resident in HBM; the batch (16 x 32 MiB = 512 MiB) is
larger than the 126 MB L2.

  value  Sum(N * ncycle) / time, fields resident in HBM, timed with CUDA events on the
         library's stream, max over ranks
  e2e    the same step (the batch of realizations, ten spans) through the C-ABI call pmx_link_run on HOST buffers
         (pinned): plan and device field created, H2D of every realization's field, the spans, D2H, all inside
         the timed call.  e2e.script_flow: one realization through the reference's own script calls --
         GSTATE.FIELDX/Y assigned from host arrays, fiber(x,'gps-') + ampliflat() per span, GSTATE.FIELDX/Y
         read back (e2e_per_call: H2D and D2H inside every fiber()/ampliflat() call)
  roofline      dominant pass kernel: 64 algorithmic bytes per live Sa and step / its device time
                (CUDA events around every launch of one extra, profiled link pass)
  mc            Monte-Carlo BER leg (BASELINE config C5): --mc-realizations (default 1024) realizations of the C2 link
                in TOTAL, sharded over the ranks (strong scaling): link + equaliser + on-GPU error count + integer
                all-reduce; fields, plans and buffers are created before the clock starts
  configs       one span of every other BASELINE configuration on a resident batch, CUDA events on the library's
                stream: C1 (batch 1 and 64), C3 ('gp--' against the FP64 roofline, and 'gps-'), C4 -- each with its
                own roofline fraction
  cpu_baseline  the numpy oracle (op-for-op restatement of fiber.m) on one host core, on a
                bounded sample of the same workload: span 1 of the link (80 km, 100 plates) at full N

--impl reference times the CPU path (oracle port; no Octave/MATLAB exists in the image) with
one worker process per host core, each on its own realization; a step is span 1 of the link
(config.cpu_sample says so).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NSYMB, NT, RATE, PAVG = 1 << 16, 16, 28.0, 2.0
NSPAN, SPAN_KM, NPLATES, DGD = 10, 80.0, 100, 0.1
GAIN_DB, NF_DB = 16.0, 5.0
ALG_BYTES_PER_SA_STEP = 192.0   # 3 passes x (read + write) x 32 B   (SURVEY 8d)
# dram__bytes_read.sum + dram__bytes_write.sum per Sa of a launch, from the ncu --set full capture summarised in
# profiles/r2_ncu_final_summary.txt (batch 16 in two groups: 8 realizations of 2^20 Sa per launch): pass A
# (271.3+209.2) MB, B (269.5+219.7) MB, C (271.2+208.7) MB  ->  bytes per Sa; below the 64 algorithmic bytes because
# part of the traffic is served by the L2
NCU_DRAM_BYTES_PER_SA = {'passA': 480.5e6 / (8 << 20), 'passB': 489.1e6 / (8 << 20), 'passC': 480.0e6 / (8 << 20)}
CPU_SAMPLE_KM = SPAN_KM         # bounded CPU sample: span 1 of the link in full (80 km, 100 plates): 15-30 s per core
# FP64 work of one whole trunk on one Sa (both polarizations of a bin) as pass B executes it: phasor progression 1 complex
# product, phasor on one polarization 1 complex product (2 mul + 2 fma each), boundary matrix 4 mul + 8 fma
# ->  20 FP64 instructions = 32 flops; used for the FP64 roofline of the one-step 'gp--' run of C3
FLOPS_PER_SA_TRUNK = 32.0
FP64_INSTR_PER_SA_TRUNK = 20.0
FP64_FMA_PER_CLK_SM = 64.0      # measured: tools/ubench/fp64_rate.cu, 63.9 DFMA/clk/SM on this B200
# FP64 instructions (DFMA + DADD + DMUL) per Sa of a launch, from the same ncu capture: sm__pipe_fp64_cycles_active x 2 warp
# instructions per active cycle and SM x 32 threads / (Sa per SM); pass B also counted instruction by instruction on the
# source page (214.6).  The FP64-pipe floor of a pass = this / (64 per clock and SM x 148 SMs x SM clock).
NCU_FP64_INSTR_PER_SA = {'passA': 94.9, 'passB': 214.6, 'passC': 82.8}


def fiber_params(length_m, nplates):
    from polmux_b200 import synth
    f = dict(synth.SMF)
    f.update(length=length_m, dgd=DGD, nplates=nplates, manakov='yes')
    return f


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                      '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5).stdout
                self.samples.append([v.strip() for v in out.strip().split(',')])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = [float(s[0]) for s in self.samples if len(s) >= 6 and s[0].replace('.', '').isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) >= 6 and s[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({names[i] for s in self.samples if len(s) >= 6 for i in range(4) if s[2 + i] == 'Active'})
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(sm)}


# ----------------------------------------------------------------------------------------
def cpu_sample(seed):
    """One bounded CPU sample: span 1 (CPU_SAMPLE_KM) at full N through the oracle.
    -> (Sa*steps, seconds)."""
    import oracle.fiber_oracle as orc
    from polmux_b200 import synth
    ex, ey, _, _ = synth.pdm_qpsk(NSYMB, NT, 1)
    gs = orc.reset_all(NSYMB, NT, 1)
    gs.SYMBOLRATE, gs.LAMBDA, gs.POWER = RATE, np.array([1550.0]), np.array([PAVG])
    orc.create_field(gs, 'unique', ex, ey, power_average=True)
    npl = int(round(NPLATES * CPU_SAMPLE_KM / SPAN_KM))
    fib = fiber_params(CPU_SAMPLE_KM * 1e3, npl)
    t0 = time.perf_counter()
    orc.fiber(gs, fib, 'gps-', rng=np.random.Generator(np.random.PCG64(seed)))
    dt = time.perf_counter() - t0
    return float(NSYMB * NT) * gs.log['ncycle'], dt


def _cpu_worker(seed):
    os.environ.setdefault('OMP_NUM_THREADS', '1')
    return cpu_sample(seed)


def run_reference(args, rank, world, out=sys.stdout):
    """--impl reference: the CPU SSFM on all host cores (one realization per worker process)."""
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    sample = ('span 1 of %d (%.0f km, %d plates, no amplifier) at N=2^20, one realization per worker, %d workers'
              % (NSPAN, CPU_SAMPLE_KM, int(round(NPLATES * CPU_SAMPLE_KM / SPAN_KM)), cores))
    ctx = mp.get_context('spawn')
    with ctx.Pool(cores) as pool:
        for w in range(min(args.warmup, 1)):     # numpy has nothing to warm up beyond the first call
            pool.map(_cpu_worker, [1000 + i for i in range(cores)])
        t0 = time.perf_counter()
        work = 0.0
        for k in range(args.steps):
            res = pool.map(_cpu_worker, [1000 + i for i in range(cores)])
            work += sum(r[0] for r in res)
        dt = time.perf_counter() - t0
    val = work / dt / 1e9
    line = {'impl': 'reference', 'metric': 'ssfm_gsa_steps_per_s', 'value': val, 'unit': 'GSa*steps/s',
            'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': dt / max(args.steps, 1) * 1e3, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': dict(workload_config(args, world), cpu_sample=sample, cpu_sample_spans=1, cpu_sample_km=CPU_SAMPLE_KM,
                           realizations_per_step=cores),
            'cpu_baseline': {'value': val, 'unit': 'GSa*steps/s', 'cores': cores, 'kind': 'port', 'sample': sample},
            'e2e': {'value': val, 'unit': 'GSa*steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    out.write(json.dumps(line) + "\n")
    out.flush()


def workload_config(args, world):
    return {'workload': 'C2', 'nfft': NSYMB * NT, 'spans': NSPAN, 'span_km': SPAN_KM, 'flag': 'gps-',
            'manakov': 'yes', 'nplates': NPLATES, 'dgd_symbols': DGD, 'ampli_gain_db': GAIN_DB, 'ampli_f_db': NF_DB,
            'pavg_mw': PAVG, 'symbolrate_gbaud': RATE, 'realizations_per_gpu': args.batch,
            'l2_policy': 'batch working set %d MiB > 126 MB L2' % (args.batch * 32),
            'parallelism': 'realizations sharded over %d GPU(s), no data-path collective' % world}


# ----------------------------------------------------------------------------------------
CONFIG_CASES = [  # key, description, nsymb, nt, nch, mW per channel, fiber overrides, flag, batch
    ('C1_batch1', 'Run_my_PDM_QPSK: 2^16 Sa, 100 km, CNLSE, 10 plates, one realization',
     1 << 12, 16, 1, 2.0, dict(length=1e5, dgd=1.0, nplates=10, manakov='no'), 'gps-', 1),
    ('C1_batch64', 'Run_my_PDM_QPSK, 64 realizations resident',
     1 << 12, 16, 1, 2.0, dict(length=1e5, dgd=1.0, nplates=10, manakov='no'), 'gps-', 64),
    ('C3_gp', "ex24_pmd with the reference's flag 'gp--': one linear step of 200 trunks, DGD 0.5 symbol, 8 realizations",
     1 << 16, 16, 1, 2.0, dict(length=8e4, dgd=0.5, nplates=200), 'gp--', 8),
    ('C3_gps', "ex24_pmd fiber with 'gps-' (Manakov), 200 plates per span, 8 realizations",
     1 << 16, 16, 1, 2.0, dict(length=8e4, dgd=0.5, nplates=200, manakov='yes'), 'gps-', 8),
    ('C4', 'nine 28-GBaud channels in one field of 2^22 Sa, 80 km Manakov, 1 mW per channel, 2 realizations',
     1 << 16, 64, 9, 1.0, dict(length=8e4, dgd=0.1, nplates=100, manakov='yes'), 'gps-', 2),
]


def config_legs(ctx, stream, torch, peak, peaks):
    """One span of every BASELINE configuration besides the headline one, on a resident batch: best of 3 runs, CUDA
    events on the library's stream.  'gp--' (one step, 200 trunks per Sa) is bound by the FP64 pipe, not by HBM: it is
    reported against 2*64*148*f_max flop/s (64 DFMA per clock and SM measured, tools/ubench/fp64_rate.cu)."""
    import polmux_b200 as pmx
    from polmux_b200 import _lib, mc, synth
    from polmux_b200.fiber import fiber_setup, setup_to_desc
    out = {}
    fmax = float(peaks.get('sm_max_mhz', 1965.0)) * 1e6
    fp64_peak = 2.0 * FP64_FMA_PER_CLK_SM * 148 * fmax / 1e12
    for key, what, nsymb, nt, nch, pw, over, flag, B in CONFIG_CASES:
        N = nsymb * nt
        ex, ey, _, _ = synth.pdm_qpsk(nsymb, nt, nch)
        pmx.reset_all(nsymb, nt, nch)
        G = pmx.GSTATE
        G.SYMBOLRATE, G.LAMBDA, G.POWER = RATE, synth.wdm_lambdas(nch, 1550.0, 0.4), np.full(nch, pw)
        pmx.create_field('unique', ex, ey, {'power': 'average'})
        fib = dict(synth.SMF)
        fib.update(over)
        setup = fiber_setup(fib, flag, rng=np.random.Generator(np.random.PCG64(0)))
        d = [mc.draw_plates(1000 + b, setup.nplates) for b in range(B)]
        pl = [np.stack([x[i] for x in d]) for i in range(3)]
        desc, keep = setup_to_desc(setup, batch=B, plate_sets=B, db0=pl[0], theta=pl[1], epsilon=pl[2])
        plan = _lib.Plan(ctx, desc, keep)
        tx = _lib.DeviceField(ctx, N, 1, 1)
        tx.upload(G.FIELDX, G.FIELDY)
        work = _lib.DeviceField(ctx, N, 1, B)
        best, res = None, None
        for rep in range(4):                         # the first run is the warm-up
            work.broadcast_from(tx)
            ctx.sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            res = plan.execute(work)
            e1.record(stream)
            ctx.sync()
            ms = e0.elapsed_time(e1)
            if rep > 0:
                best = ms if best is None else min(best, ms)
        sa = float(res.ncycle.sum()) * N
        v = sa / (best * 1e-3) / 1e9
        item = {'what': what, 'nfft': N, 'batch': B, 'flag': flag, 'ncycle': int(res.ncycle[0]), 'ms_per_span': best,
                'value': v, 'unit': 'GSa*steps/s',
                'roofline': {'bound': 'hbm', 'achieved': ALG_BYTES_PER_SA_STEP * v, 'peak': peak, 'unit': 'GB/s',
                             'frac': ALG_BYTES_PER_SA_STEP * v / peak}}
        if flag == 'gp--':
            trunks = float(setup.nplates) * B * N / (best * 1e-3)
            tf = trunks * FLOPS_PER_SA_TRUNK / 1e12
            item['gsa_trunks_per_s'] = trunks / 1e9
            item['roofline'] = {'bound': 'fp64', 'achieved': tf, 'peak': fp64_peak, 'unit': 'TFLOP/s', 'frac': tf / fp64_peak,
                                'flops_per_sa_trunk': FLOPS_PER_SA_TRUNK, 'fp64_instr_per_sa_trunk': FP64_INSTR_PER_SA_TRUNK,
                                'fp64_issue_frac': trunks * FP64_INSTR_PER_SA_TRUNK / (FP64_FMA_PER_CLK_SM * 148 * fmax),
                                'peak_source': '2 * 64 DFMA/clk/SM (measured) * 148 SMs * sm_max_mhz'}
        out[key] = item
        for f in (tx, work):
            f.close()
        plan.close()
    return out


DUMP_SAMPLES = 1 << 16     # per realization and polarization: 2 x 16 x 2^16 x 16 B = 32 MiB for the default batch
DUMP_FIELD_BYTES = 48 << 20   # larger batches get fewer samples so that a dump stays below 64 MB
DUMP_SEED = 20240601


def dump_outputs(d, work, link):
    """What the timed step hands its caller, from the last timed step: the received field of every realization and
    the number of SSFM steps each span took.  The field (32 MiB per realization) is sampled at DUMP_SAMPLES indices
    drawn once from a fixed seed, the same in every run, so that two builds can be compared output for output:
      field_x.npy, field_y.npy  float64 [batch, S, 2]  (real, imaginary) at the S sampled indices
      sample_index.npy          float64 [S]            the indices into the 2^20 samples of a realization
      ncycle.npy                float64 [spans, batch] steps per span and realization"""
    os.makedirs(d, exist_ok=True)
    n = work.nfft
    ns = min(DUMP_SAMPLES, n, DUMP_FIELD_BYTES // (32 * work.batch))
    idx = np.sort(np.random.Generator(np.random.PCG64(DUMP_SEED)).choice(n, ns, replace=False))
    fx = np.empty((work.batch, idx.size, 2))
    fy = np.empty_like(fx)
    for b in range(work.batch):                    # one realization at a time keeps the host copy at 32 MiB
        x, y = work.download(b0=b, nb=1)
        for out, f in ((fx, x), (fy, y)):
            out[b, :, 0], out[b, :, 1] = f[0, 0, idx].real, f[0, 0, idx].imag
    np.save(os.path.join(d, 'field_x.npy'), fx)
    np.save(os.path.join(d, 'field_y.npy'), fy)
    np.save(os.path.join(d, 'sample_index.npy'), idx.astype(np.float64))
    np.save(os.path.join(d, 'ncycle.npy'), np.array(link.ncycles, dtype=np.float64))


def _claim_stdout():
    """Keep stdout for the one JSON line: libraries (NCCL's version banner, torchrun notices) that write to
    file descriptor 1 are redirected to stderr; returns a writer bound to the original stdout."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(real, 'w')


def main():
    out = _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--batch', type=int, default=16, help='realizations per GPU per step')
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-mc', action='store_true')
    ap.add_argument('--no-fp32', action='store_true', help='skip the separately reported FP32 leg')
    ap.add_argument('--mc-realizations', type=int, default=1024,
                    help='Monte-Carlo leg (C5): realizations in TOTAL over all ranks (strong scaling)')
    ap.add_argument('--no-configs', action='store_true', help='skip the per-configuration legs (C1, C3, C4)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help="write rank 0's output of the last timed step to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        run_reference(args, rank, world, out)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    import polmux_b200 as pmx
    from polmux_b200 import _lib, synth
    from polmux_b200.fiber import fiber_setup, setup_to_desc

    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    ctx = _lib.Context(local)
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device('cuda', local))

    # ---- Tx field (host, seeded) and fiber set-up
    N = NSYMB * NT
    ex, ey, symx, symy = synth.pdm_qpsk(NSYMB, NT, 1)
    pmx.reset_all(NSYMB, NT, 1)
    G = pmx.GSTATE
    G.SYMBOLRATE, G.LAMBDA, G.POWER = RATE, np.array([1550.0]), np.array([PAVG])
    pmx.create_field('unique', ex, ey, {'power': 'average'})
    fib = fiber_params(SPAN_KM * 1e3, NPLATES)
    setup = fiber_setup(fib, 'gps-', rng=np.random.Generator(np.random.PCG64(0)))
    B = args.batch

    # realization r (global index) of span k draws its plates from seed 1000 + r + 100000*k (polmux_b200.mc)
    from polmux_b200 import mc
    link = mc.Link(ctx, setup, NSPAN, B, GAIN_DB, NF_DB, first_realization=rank * B)
    tx = _lib.DeviceField(ctx, N, 1, 1)
    tx.upload(G.FIELDX, G.FIELDY)
    work = _lib.DeviceField(ctx, N, 1, B)

    def link_step(step_id):
        """one pass of the 10-span link over the resident batch -> Sa*steps done"""
        work.broadcast_from(tx)
        return link.run(work, ase_seed=step_id)

    def barrier():
        ctx.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ctx.sync()

    for w in range(args.warmup):
        link_step(w)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    total = 0
    for k in range(args.steps):
        total += link_step(100 + k)
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    gpu_launches = ctx.launches - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, work, link)
    sampler.stop_flag = True
    t = torch.tensor([ms, float(total)], dtype=torch.float64, device='cuda')
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        ms, total_all = float(tmax[0]), float(tsum[1])
    else:
        total_all = float(total)
    value = total_all / (ms * 1e-3) / 1e9

    # ---- per-pass timing (separate, profiled pass over one link step; events around every launch)
    ctx.profile(True)
    prof_sa_steps = link_step(999)
    pms, pn = ctx.profile_read()
    ctx.profile(False)
    roof = None
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak = float(peaks.get('hbm_gbs', 6650.0))
    peak_src = 'measured (MEASURED_PEAKS.json hbm_gbs)' if 'hbm_gbs' in peaks else 'fallback 6650 GB/s (B200_PROFILING.md)'
    if pn[1] > 0:
        names = ['passA', 'passB', 'passC']
        dom = int(np.argmax(pms[:3]))
        # every live Sa is read and written once per pass and per step: 64 algorithmic bytes.  Launches
        # that find their realizations finished exit at once; they count as launches, not as bytes.
        alg_bytes = 64.0 * prof_sa_steps
        ach = alg_bytes / (pms[dom] * 1e-3) / 1e9
        roof = {'bound': 'hbm', 'kernel': names[dom], 'achieved': ach, 'peak': peak, 'unit': 'GB/s',
                'frac': ach / peak, 'traffic': NCU_DRAM_BYTES_PER_SA[names[dom]] * prof_sa_steps / float(pn[dom]),
                'traffic_source': 'ncu --set full, profiles/r2_ncu_final_summary.txt, scaled to the Sa of a launch',
                'peak_source': peak_src,
                'bytes_per_launch': alg_bytes / float(pn[dom]), 'ms_per_launch': pms[dom] / float(pn[dom]),
                'launches_timed': int(pn[dom]),
                'pass_share_of_step': {names[i]: float(pms[i] / pms[:3].sum()) for i in range(3)},
                'pass_gbs': {names[i]: alg_bytes / (pms[i] * 1e-3) / 1e9 for i in range(3)}}
    step_roof = {'achieved': ALG_BYTES_PER_SA_STEP * value / world, 'peak': peak, 'unit': 'GB/s',
                 'frac': ALG_BYTES_PER_SA_STEP * value / world / peak, 'bytes_per_sa_step': ALG_BYTES_PER_SA_STEP,
                 'per': 'GPU'}

    # ---- FP32 mode, reported separately (north_star): same link, fields and arithmetic in float
    fp32 = None
    if not args.no_fp32:
        link32 = mc.Link(ctx, setup, NSPAN, B, GAIN_DB, NF_DB, first_realization=rank * B, precision='f32')
        tx32 = _lib.DeviceField(ctx, N, 1, 1, precision=_lib.PMX_F32)
        tx32.upload(G.FIELDX, G.FIELDY)
        work32 = _lib.DeviceField(ctx, N, 1, B, precision=_lib.PMX_F32)

        def link32_step(step_id):
            work32.broadcast_from(tx32)
            return link32.run(work32, ase_seed=step_id)

        for w in range(min(args.warmup, 2)):
            link32_step(w)
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(stream)
        tot32 = 0
        for k in range(args.steps):
            tot32 += link32_step(100 + k)
        f1.record(stream)
        barrier()
        t32 = torch.tensor([f0.elapsed_time(f1), float(tot32)], dtype=torch.float64, device='cuda')
        if world > 1:
            a = t32.clone()
            dist.all_reduce(a, op=dist.ReduceOp.MAX)
            b = t32.clone()
            dist.all_reduce(b, op=dist.ReduceOp.SUM)
            t32 = torch.stack([a[0], b[1]])
        v32 = float(t32[1]) / (float(t32[0]) * 1e-3) / 1e9
        # accuracy of the mode on this workload: span 1 (no ASE) of realization 0, FP32 against FP64
        one64 = _lib.DeviceField(ctx, N, 1, 1)
        one32 = _lib.DeviceField(ctx, N, 1, 1, precision=_lib.PMX_F32)
        one64.upload(G.FIELDX, G.FIELDY)
        one32.upload(G.FIELDX, G.FIELDY)
        pl0 = mc.draw_plates(mc.plate_seed(0, 0), NPLATES)
        errs = []
        outs = []
        for prec, fld in (('f64', one64), ('f32', one32)):
            d1, k1 = setup_to_desc(setup, batch=1, plate_sets=1, db0=pl0[0][None], theta=pl0[1][None], epsilon=pl0[2][None],
                                   precision=prec)
            pl = _lib.Plan(ctx, d1, k1)
            pl.execute(fld)
            outs.append(fld.download())
            pl.close()
        num = np.sqrt(np.sum(np.abs(outs[1][0] - outs[0][0]) ** 2) + np.sum(np.abs(outs[1][1] - outs[0][1]) ** 2))
        den = np.sqrt(np.sum(np.abs(outs[0][0]) ** 2) + np.sum(np.abs(outs[0][1]) ** 2))
        fp32 = {'value': v32, 'unit': 'GSa*steps/s', 'dtype': 'f32', 'ms_per_step': float(t32[0]) / max(args.steps, 1),
                'bytes_per_sa_step': ALG_BYTES_PER_SA_STEP / 2, 'roofline_step_frac': ALG_BYTES_PER_SA_STEP / 2 * v32 / world / peak,
                'rel_l2_vs_f64_one_span': float(num / den), 'tolerance': 1e-5}
        del link32, work32, tx32, one64, one32

    # ---- Monte-Carlo BER leg (config C5, bounded): link + linear equaliser + on-GPU error counter,
    # counts all-reduced over the ranks (NCCL), ber_estimate's recursion replayed on the host
    mcres = None
    if not args.no_mc:
        sym = np.stack([symx[:, 0], symy[:, 0]]).astype(np.uint8)
        nreal = max(int(args.mc_realizations), world)
        # fields, the link and equaliser plans, twiddle tables and count buffers are created here, outside the clock;
        # one untimed pass over a single group per rank warms them up
        warm = mc.McRunner(ctx, setup, G.FIELDX_TX, G.FIELDY_TX, sym, NSYMB, NT, NSPAN, GAIN_DB, NF_DB, B * world, B,
                           rank, world)
        warm.run(ase_seed=7)
        warm.close()
        runner = mc.McRunner(ctx, setup, G.FIELDX_TX, G.FIELDY_TX, sym, NSYMB, NT, NSPAN, GAIN_DB, NF_DB, nreal, B,
                             rank, world)
        runner.work.broadcast_from(runner.tx)
        runner.link.equalize(runner.work)            # builds the equaliser plan (the field is overwritten by run())
        barrier()
        t0 = time.perf_counter()
        counts, _ = runner.run(ase_seed=7)
        barrier()
        tdt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(tdt, op=dist.ReduceOp.MAX)
        runner.close()
        rep = mc.ber_replay(counts, 4 * NSYMB, stop=(0.1, 68.0), nmin=100)
        mcres = {'realizations_per_s': nreal / float(tdt[0]), 'realizations': nreal, 'seconds': float(tdt[0]),
                 'scaling': 'strong', 'realizations_per_rank': (nreal + world - 1) // world,
                 'timing': 'one pass over all realizations, host clock between barriers, max over ranks; allocations, '
                           'plans and a warm-up group outside',
                 'errors_total': int(counts.sum()), 'bits_per_realization': 4 * NSYMB, 'avgber': rep['avgber'],
                 'count_reduce': 'all_reduce(int64[%d], sum) over %d rank(s), backend %s'
                                 % (nreal, world, 'nccl' if world > 1 else 'none (single rank)'),
                 'receiver': 'genie: ideal linear equaliser from the known plates + data-aided decision'}
        # the same job with the reference's receive chain behind the link (receiver_cohmix front-end, sampler, CMA
        # polarization demultiplexer, Viterbi & Viterbi, differential decision), on a bounded number of realizations; the
        # chain of a group runs on its own stream beside the propagation of the next group (plans created by McRunner)
        nrx = max(B * world, min(nreal, 8 * B * world if world == 1 else 4 * B * world))
        rxr = mc.McRunner(ctx, setup, G.FIELDX_TX, G.FIELDY_TX, sym, NSYMB, NT, NSPAN, GAIN_DB, NF_DB, nrx, B, rank, world,
                          receiver='cohmix')
        barrier()
        t0 = time.perf_counter()
        rxc, _ = rxr.run(ase_seed=7)
        barrier()
        tdx = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(tdx, op=dist.ReduceOp.MAX)
        npass = [int(p.max()) for p in rxr.passes]
        rxr.close()
        mcres['receiver_chain'] = {'receiver': "cohmix: receiver_cohmix front-end (gauss 1.9 / bessel5 0.65) + sampler + CMA + "
                                               'Viterbi & Viterbi + differential decision, all on the device',
                                   'realizations': nrx, 'seconds': float(tdx[0]), 'realizations_per_s': nrx / float(tdx[0]),
                                   'errors_total': int(rxc.sum()), 'cma_passes_max_rank0': max(npass) if npass else 0,
                                   # a constant-modulus demultiplexer started from the identity can lock both outputs on the
                                   # same polarization (the reference's cmapolardemux does the same; its scripts run with
                                   # applypol = false): those realizations count about half the bits of one polarization
                                   'cma_singular_realizations': int((rxc > NSYMB // 2).sum()),
                                   'errors_without_singular': int(rxc[rxc <= NSYMB // 2].sum())}

    # ---- e2e: the reference's own script flow on HOST buffers (one realization, all spans):
    #   GSTATE.FIELDX/FIELDY <- pinned host arrays; for each span fiber(x,'gps-'), ampliflat(G,'gain',opt); read the
    #   received field out of GSTATE.  The field crosses PCIe once in and once out per link (the library keeps it in
    #   HBM between the in-line devices, polmux_b200/gstate.py); e2e_per_call = the same calls with a download and an
    #   upload in every fiber() and ampliflat(), i.e. what a stateless MEX gateway pays.
    e2e = None
    e2e_pc = None
    if not args.no_e2e:
        from polmux_b200 import gstate
        pinx = torch.empty((N, 1), dtype=torch.complex128).pin_memory()
        piny = torch.empty((N, 1), dtype=torch.complex128).pin_memory()
        txx, txy = np.array(G.FIELDX_TX), np.array(G.FIELDY_TX)

        def e2e_step(sid):
            """-> (Sa*steps, seconds).  The clock starts with the Tx field in the pinned host arrays and stops when
            the Rx field is back in them: H2D, ten spans, D2H.  (Refilling the arrays with the Tx field for the next
            step is the harness's business and stays outside.)"""
            hx, hy = pinx.numpy(), piny.numpy()
            hx[...] = txx
            hy[...] = txy
            ctx.sync()
            t0 = time.perf_counter()
            G.FIELDX, G.FIELDY = hx, hy
            G.DELAY, G.DISP = np.zeros((2, 1)), np.zeros((2, 1))
            sa = 0
            for k in range(NSPAN):
                pmx.fiber(fib, 'gps-', rng=np.random.Generator(np.random.PCG64(1000 + rank + 100000 * k)), ctx=ctx)
                sa += pmx.FIBER_LAST['ncycle'] * N
                pmx.ampliflat(GAIN_DB, 'gain', {'f': NF_DB}, ctx=ctx, seed=sid * 64 + k)
            rx, ry = G.FIELDX, G.FIELDY      # the step's result, read on the host (D2H of both polarizations)
            ctx.sync()
            dt = time.perf_counter() - t0
            assert rx is hx and ry is hy and np.isfinite(rx[0, 0]) and not G.is_resident()
            return sa, dt

        def e2e_leg(resident, nsteps):
            gstate.RESIDENT = resident
            try:
                for w in range(2):
                    e2e_step(w)
                barrier()
                sa, dt = 0, 0.0
                for k in range(nsteps):
                    a, b = e2e_step(10 + k)
                    sa += a
                    dt += b
            finally:
                gstate.RESIDENT = True
            tt = torch.tensor([dt, float(sa)], dtype=torch.float64, device='cuda')
            if world > 1:
                a = tt.clone()
                dist.all_reduce(a, op=dist.ReduceOp.MAX)
                b = tt.clone()
                dist.all_reduce(b, op=dist.ReduceOp.SUM)
                return float(b[1]) / float(a[0]) / 1e9
            return sa / dt / 1e9

        per_field = N * 32
        ne2e = max(2, args.steps)
        e2e_script = {'value': e2e_leg(True, ne2e), 'unit': 'GSa*steps/s',
                      'h2d_bytes_per_step': per_field, 'd2h_bytes_per_step': per_field,
                      'api': "GSTATE.FIELDX/Y <- pinned host field; 10 x [fiber(x,'gps-'); ampliflat(G,'gain',opt)]; read "
                             "GSTATE.FIELDX/Y (field resident in HBM between the calls), 1 realization per rank"}

        # the step of `value` (B realizations x 10 spans) through the C-ABI call on HOST buffers: pmx_link_run creates the
        # plan and the device field, uploads the B fields, loops the spans, downloads the B fields and frees everything
        import ctypes as _C
        bx = torch.empty((B, 1, N), dtype=torch.complex128).pin_memory()
        by = torch.empty((B, 1, N), dtype=torch.complex128).pin_memory()
        txr, tyr = np.ascontiguousarray(txx.T), np.ascontiguousarray(txy.T)       # [1][N]
        lk = mc.Link(ctx, setup, NSPAN, B, GAIN_DB, NF_DB, first_realization=rank * B)   # (plate draws and sigma only)
        desc_b, keep_b = setup_to_desc(setup, batch=B, plate_sets=B, db0=lk.plates[0][0], theta=lk.plates[0][1],
                                       epsilon=lk.plates[0][2])

        def e2e_batched(sid):
            hx, hy = bx.numpy(), by.numpy()
            hx[...] = txr[None]
            hy[...] = tyr[None]
            ldesc, lkeep = _lib.make_link(NSPAN, lk.gain, lk.sigma,
                                          plates=[np.stack([pl[i] for pl in lk.plates]) for i in range(3)], plate_sets=B,
                                          seeds=[lk.ase_seed(sid, k) for k in range(NSPAN)], first=rank * B)
            io = _lib.complex_field(hx, hy)
            res = _lib.Result(NSPAN * B)
            ctx.sync()
            t0 = time.perf_counter()
            ctx.check(ctx.lib.pmx_link_run(ctx.h, _C.byref(desc_b), _C.byref(ldesc), _C.byref(io), _C.byref(res.c)))
            dt = time.perf_counter() - t0
            assert np.isfinite(hx[B - 1, 0, 0]) and not np.array_equal(hx[0, 0, :8], txr[0, :8])
            return int(res.ncycle.sum()) * N, dt

        for w in range(2):
            e2e_batched(w)
        barrier()
        sa_b, dt_b = 0, 0.0
        for k in range(ne2e):
            a, b_ = e2e_batched(10 + k)
            sa_b += a
            dt_b += b_
        tt = torch.tensor([dt_b, float(sa_b)], dtype=torch.float64, device='cuda')
        if world > 1:
            a = tt.clone()
            dist.all_reduce(a, op=dist.ReduceOp.MAX)
            b_ = tt.clone()
            dist.all_reduce(b_, op=dist.ReduceOp.SUM)
            v_b = float(b_[1]) / float(a[0]) / 1e9
        else:
            v_b = sa_b / dt_b / 1e9
        e2e = {'value': v_b, 'unit': 'GSa*steps/s', 'h2d_bytes_per_step': B * per_field, 'd2h_bytes_per_step': B * per_field,
               'api': 'pmx_link_run(ctx, fiber desc, link desc, HOST fields, result) -- the C-ABI call: %d realizations per '
                      'rank in pinned host buffers, plan + device field created, H2D, 10 x [fiber ; ampliflat], D2H, all '
                      'inside the timed call (wall clock)' % B,
               'script_flow': e2e_script}
        lk.plan.close()
        del bx, by
        # a stateless gateway: fiber() and ampliflat() each copy the field up and down
        e2e_pc = {'value': e2e_leg(False, 2), 'unit': 'GSa*steps/s',
                  'h2d_bytes_per_step': NSPAN * 2 * per_field, 'd2h_bytes_per_step': NSPAN * 2 * per_field,
                  'api': 'the same calls with gstate.RESIDENT = False (H2D + D2H inside every call)'}

    # ---- the other BASELINE configurations, one span each on a resident batch (every rank runs them so that the ranks
    # stay in step, the figures are rank 0's); last of the GPU legs: they re-initialise GSTATE with their own sizes)
    cfgs = None
    if not args.no_configs:
        cfgs = config_legs(ctx, stream, torch, peak, peaks)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        sa, dt = cpu_sample(1000)
        cpu = {'value': sa / dt / 1e9, 'unit': 'GSa*steps/s', 'cores': 1, 'kind': 'port',
               'sample': 'span 1 of %d (%.0f km, %d plates, no amplifier) at N=2^20, 1 realization, numpy oracle (%.1f s)'
                         % (NSPAN, CPU_SAMPLE_KM, int(round(NPLATES * CPU_SAMPLE_KM / SPAN_KM)), dt)}

    if rank == 0:
        sampler.join(timeout=2)
        clk = sampler.summary()
        if roof and clk.get('sm_mhz'):
            # the second ceiling of the dominant pass on this part: 64 FP64 instructions per clock and SM
            fl = NCU_FP64_INSTR_PER_SA[roof['kernel']] / (FP64_FMA_PER_CLK_SM * 148 * clk['sm_mhz'] * 1e6)   # s per Sa
            t_sa = 64.0 / (roof['achieved'] * 1e9)
            roof['fp64_pipe'] = {'instr_per_sa': NCU_FP64_INSTR_PER_SA[roof['kernel']], 'floor_ps_per_sa': fl * 1e12,
                                 'hbm_floor_ps_per_sa': 64.0 / (roof['peak'] * 1e9) * 1e12, 'measured_ps_per_sa': t_sa * 1e12,
                                 'frac_of_fp64_floor': fl / t_sa,
                                 'note': 'FP64 pipe floor at the SM clock sampled during the run; above the HBM floor for pass B'}
        line = {'metric': 'ssfm_gsa_steps_per_s', 'value': value, 'unit': 'GSa*steps/s', 'n_gpus': world,
                'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms / max(args.steps, 1),
                'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64',
                'data': 'synthetic', 'config': workload_config(args, world), 'clocks': sampler.summary(),
                'e2e': e2e, 'e2e_per_call': e2e_pc, 'gpu_launches': int(gpu_launches), 'roofline': roof, 'roofline_step': step_roof,
                'cpu_baseline': cpu, 'mc': mcres, 'configs': cfgs, 'fp32': fp32,
                'sa_steps_per_step': total_all / max(args.steps, 1)}
        out.write(json.dumps(line) + '\n')
        out.flush()
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
