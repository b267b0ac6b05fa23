"""Batched Monte-Carlo over independent realizations: the one axis the path shards on.

The reference runs realizations one after another in `while cond` loops
(ex20_coherent_polmux.m:131-181) and feeds the integer error count of each block to
ber_estimate (ber_estimate.m:118).  Here a group of realizations (same Tx field, different
waveplate draws and ASE seeds) is resident in HBM and advances through the whole link --
nspan x [fiber(x,'gps-') ; ampliflat(G,'gain',{f})] -- without returning to the host; groups
are sharded contiguously over the ranks (one process per GPU) and the only collective is an
integer all-reduce (NCCL) of the per-realization error counts.  The host then replays
ber_estimate's order-dependent recursion in realization order, so the estimate is the same
whatever the number of GPUs.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Optional

import numpy as np

from . import _lib
from .ampliflat import ase_sigma
from .fiber import FiberSetup, setup_to_desc


def draw_plates(seed: int, nplates: int):
    """fiber.m:274-276 with the stream of one realization/span."""
    r = np.random.Generator(np.random.PCG64(int(seed)))
    db0 = r.random(nplates) * 2 * np.pi - np.pi
    theta = r.random(nplates) * np.pi - 0.5 * np.pi
    eps = 0.5 * np.arcsin(r.random(nplates) * 2 - 1)
    return db0, theta, eps


def plate_seed(realization: int, span: int) -> int:
    return 1000 + int(realization) + 100000 * int(span)


def shard(nreal: int, rank: int, world: int):
    """contiguous realization groups: rank g owns [floor(g*n/G), floor((g+1)*n/G))  (SURVEY 8e)"""
    return (rank * nreal) // world, ((rank + 1) * nreal) // world


class Link:
    """nspan identical spans resident on one GPU, for a batch of realizations."""

    def __init__(self, ctx: _lib.Context, setup: FiberSetup, nspan: int, batch: int, gain_db: float,
                 nf_db: Optional[float], first_realization: int = 0, precision: str = 'f64'):
        self.ctx, self.setup, self.nspan, self.batch = ctx, setup, nspan, batch
        self.precision = precision
        self.first = first_realization
        self.gain = 10 ** (gain_db * 0.1)
        self.sigma = ase_sigma(self.gain, nf_db, setup.nfc)
        self.plates = [self._plates(k, first_realization) for k in range(nspan)]
        desc, keep = setup_to_desc(setup, batch=batch, plate_sets=batch, db0=self.plates[0][0],
                                   theta=self.plates[0][1], epsilon=self.plates[0][2], precision=precision)
        self.plan = _lib.Plan(ctx, desc, keep)
        self._inv = None

    def _plates(self, span, first):
        d = [draw_plates(plate_seed(first + b, span), self.setup.nplates) for b in range(self.batch)]
        return tuple(np.stack([x[i] for x in d]) for i in range(3))

    def retarget(self, first_realization: int):
        """same link, next group of realizations (new plate draws)"""
        self.first = first_realization
        self.plates = [self._plates(k, first_realization) for k in range(self.nspan)]

    def run(self, field: _lib.DeviceField, ase_seed: int, noise_fn=None) -> int:
        """propagate the resident batch through every span; -> Sa*steps done.
        noise_fn(span) -> [batch][2*nfc][nfft] complex standard normals (ampliflat's options.noise,
        for parity runs); default: the device's counter-based generator keyed by (seed, span, realization)."""
        n = self.setup.nfft
        noise = None if noise_fn is None else np.stack([np.asarray(noise_fn(k), dtype=np.complex128)
                                                        for k in range(self.nspan)])
        link, keep = _lib.make_link(
            self.nspan, self.gain, self.sigma, plates=[np.stack([pl[i] for pl in self.plates]) for i in range(3)],
            plate_sets=self.batch, noise=noise, seeds=[self.ase_seed(ase_seed, k) for k in range(self.nspan)],
            first=self.first)
        res = self.plan.link_exec(field, link, keep)            # the span loop runs inside the library
        ncyc = res.ncycle.reshape(self.nspan, self.batch)
        self.ncycles = [ncyc[k].copy() for k in range(self.nspan)]
        return int(ncyc.sum()) * n * self.setup.nfc

    def ase_seed(self, ase_seed: int, span: int) -> int:
        # (the device generator is keyed by the global realization index, pmx_link_desc.realization0: the noise of a
        # realization does not depend on how the run groups or shards its realizations)
        return ((int(ase_seed) & 0xffffff) << 40) + (span << 32)

    def equalize(self, field: _lib.DeviceField):
        """Ideal linear equaliser: undo GVD and PMD of every span, last span first.  One linear
        single-step fiber per span with the plate order reversed and every phase negated
        (the inverse of prod_k R_k D_k R_k' is the same product with D_k -> D_k^-1 taken backwards,
        cf. inverse_pmd.m:100-124); attenuation was already undone by the amplifiers."""
        s = self.setup
        if self._inv is None:
            sc = dict(s.scalars)
            sc.update(b30=-sc['b30'], dgdrms=-sc['dgdrms'], beta1=-np.asarray(sc['beta1']),
                      beta2=-np.asarray(sc['beta2']))
            inv = FiberSetup(nfft=s.nfft, nfc=s.nfc, fls=(s.fls[0], s.fls[1], 0, 0), dphimaxt=math.inf,
                             dzmaxt=s.length, length=s.length, alphalin=0.0, gam=s.gam, betat=-s.betat, db1=-s.db1,
                             manakov=False, nplates=s.nplates, brf=s.brf, isv=True, isy=True, b1=s.b1, dch=s.dch,
                             scalars=sc)
            desc, keep = setup_to_desc(inv, batch=self.batch, plate_sets=self.batch, db0=-self.plates[0][0][:, ::-1],
                                       theta=self.plates[0][1][:, ::-1], epsilon=self.plates[0][2][:, ::-1])
            self._inv = _lib.Plan(self.ctx, desc, keep)
        for k in reversed(range(self.nspan)):
            db0, th, ep = self.plates[k]
            self._inv.set_plates(-db0[:, ::-1], th[:, ::-1], ep[:, ::-1], plate_sets=self.batch)
            self._inv.execute(field)

    def cd_plan(self, ctx=None):
        """the plan of cd_compensate() on `ctx` (default: the link's own context; a receive chain that runs beside the next
        group's propagation keeps its plans on a context -- a stream -- of its own)"""
        if ctx is None or ctx is self.ctx:
            if getattr(self, '_cd', None) is None:
                self._cd = self._make_cd_plan(self.ctx)
            return self._cd
        return self._make_cd_plan(ctx)

    def _make_cd_plan(self, ctx):
        s = self.setup
        sc = dict(s.scalars)
        sc.update(b30=-sc['b30'], dgdrms=0.0, beta1=-np.asarray(sc['beta1']), beta2=-np.asarray(sc['beta2']))
        total = s.length * self.nspan
        inv = FiberSetup(nfft=s.nfft, nfc=s.nfc, fls=(s.fls[0], 0, 0, 0), dphimaxt=math.inf, dzmaxt=total, length=total,
                         alphalin=0.0, gam=s.gam, betat=-s.betat, db1=np.zeros_like(s.db1), manakov=False, nplates=1,
                         brf={'db0': np.zeros(1), 'theta': np.zeros(1), 'epsilon': np.zeros(1)}, isv=True, isy=True,
                         b1=s.b1, dch=s.dch, scalars=sc)
        desc, keep = setup_to_desc(inv, batch=self.batch, plate_sets=1)
        return _lib.Plan(ctx, desc, keep)

    def cd_compensate(self, field: _lib.DeviceField):
        """What a blind receiver knows: the accumulated chromatic dispersion of the link (dsp4cohdec's p.applydcf,
        dsp4cohdec.m:200-210, as an all-pass filter): one linear step with the dispersion of all spans negated.  The PMD
        stays in the field for the polarization demultiplexer."""
        self.cd_plan().execute(field)


# ------------------------------------------------------------------------------------------
@dataclass
class BerState:
    """persistent variables of ber_estimate.m:103 (scalar case, x.dim == 1)"""
    n: int = 1
    avgber: float = 0.0
    varber: float = 0.0
    cond: bool = True


def ber_update(st: BerState, err: int, M: int, stop=(0.1, 68.0), nmin: int = 1):
    """One call of mc_run, ber_estimate.m:107-142, with the integer error count of a block of M
    bits.  -> (cond, avgber, nruns, stdber)."""
    eps = math.sqrt(2) * _erfcinv(1 - stop[1] / 100)
    nnew = st.n * M
    N = (st.n - 1) * M
    varerr = (err - err ** 2 / M) / (M - 1)
    avgerr = err / M
    st.varber = ((N - 1) * st.varber + (M - 1) * varerr + N * M / (N + M) * (st.avgber - avgerr) ** 2) / (N + M - 1)
    st.avgber = ((st.n - 1) * st.avgber + avgerr) / st.n
    stdber = math.sqrt(st.varber / (N + M))
    if eps * stdber < stop[0] * st.avgber and st.avgber * nnew >= nmin:
        st.cond = False
    st.n += 1
    return st.cond, st.avgber, (st.n - 1) * M, stdber


def _erfcinv(x):
    from scipy.special import erfcinv
    return float(erfcinv(x))


def ber_replay(counts, bits_per_realization: int, stop=(0.1, 68.0), nmin: int = 1):
    """Feed per-realization counts to the recursion in realization order; stops where the
    reference's `while cond` loop would."""
    st = BerState()
    out = None
    for k, e in enumerate(counts):
        out = ber_update(st, int(e), bits_per_realization, stop, nmin)
        if not out[0]:
            return {'avgber': out[1], 'nbits': out[2], 'stdber': out[3], 'realizations_used': k + 1, 'converged': True}
    return {'avgber': out[1], 'nbits': out[2], 'stdber': out[3], 'realizations_used': len(counts), 'converged': False}


def allreduce_counts(local_counts, r0: int, nreal: int, device=None):
    """Zero-padded [nreal] int64 vector with this rank's slice filled, summed over the ranks
    (torch.distributed: NCCL on GPUs, gloo in the CPU tests).  Integer, hence order-independent
    and bit-exact (SURVEY 8e)."""
    import torch
    import torch.distributed as dist
    if isinstance(local_counts, torch.Tensor):
        full = torch.zeros(nreal, dtype=torch.int64, device=local_counts.device)
        full[r0:r0 + local_counts.numel()] = local_counts
    else:
        full = torch.zeros(nreal, dtype=torch.int64, device=device or 'cpu')
        full[r0:r0 + len(local_counts)] = torch.as_tensor(np.asarray(local_counts, dtype=np.int64))
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(full, op=dist.ReduceOp.SUM)
    return full


class McRunner:
    """Monte-Carlo BER of `nreal` realizations sharded over `world` ranks.  Everything that is allocated or planned
    once (fields, the link and equaliser plans with their tables, the count buffers) is created here; run() is
    the job itself: plate draws of every group, broadcast of the Tx field, link, equaliser, on-GPU error count,
    integer all-reduce."""

    def __init__(self, ctx: _lib.Context, setup: FiberSetup, tx_x, tx_y, sym, nsymb: int, nt: int, nspan: int,
                 gain_db: float, nf_db: float, nreal: int, batch: int, rank: int = 0, world: int = 1,
                 receiver: str = 'genie', dsp_params=None, rx_params=None, ich: int = 1, pipeline: bool = True,
                 compensation: str = 'cd', dbp_params=None):
        """receiver: 'genie' -- ideal linear equaliser from the known plates + data-aided decision (pmx_qpsk_count);
        'blind' -- chromatic dispersion compensated, then the DSP core of dsp4cohdec (CMA polarization demultiplexer,
        Viterbi & Viterbi carrier recovery, differential decision: pmx_dsp_count, polmux_b200/dsp.py);
        'cohmix' -- chromatic dispersion compensated, the front-end of receiver_cohmix.m for channel `ich` (optical
        filter, LO mixing, photodiodes, low-pass filter; rx_params = its x struct, polmux_b200/receiver.py), the
        currents sampled at the symbol centres delayed by the filters' 'theory' delay (dsp4cohdec.m:490-503) and
        divided by 4*sqrt(POWER(ich)) (dsp4cohdec.m:226-227), then the same DSP core.
        pipeline: run the receive chain of a group beside the propagation of the next one (same counts either way)
        compensation ('blind' and 'cohmix'): 'cd' -- the all-pass step that undoes the link's dispersion; 'dbp' -- digital
        backpropagation of the link (polmux_b200/dbp.py) with dbp_params (steps_per_span, step_len, span_steps, xi; default
        one step per span, xi = 1), the amplifier gain undone before each span.  'dbp_pmd' (every receiver) -- PMD-aware
        DBP through each group's own plate draws (Link.plates); with 'genie' it replaces the linear equaliser.
        dbp_params with 'decim' (a power of two >= 2; 'blind' and 'cohmix', a one-column 'unique' field): single-channel DBP
        on nfft/decim samples -- of channel `ich` for 'cohmix', of the channel at the centre of the grid for 'blind'.
        dbp_params with 'filter_bw' [GHz]: filtered DBP (dbp_plan); with 'nl_taps': enhanced split-step DBP (dbp_plan)"""
        import torch
        from . import dsp as _dsp
        self.receiver, self.dsp_params = receiver, dict(dsp_params or {})
        if receiver not in ('genie', 'blind', 'cohmix'):
            raise ValueError("receiver must be 'genie', 'blind' or 'cohmix'")
        if compensation not in ('cd', 'dbp', 'dbp_pmd'):
            raise ValueError("compensation must be 'cd', 'dbp' or 'dbp_pmd'")
        if compensation == 'dbp' and receiver == 'genie':
            raise ValueError("the genie receiver undoes the link with the known plates: compensation='dbp' needs 'blind' or 'cohmix'")
        if receiver == 'genie' and dict(dbp_params or {}).get('decim') is not None:
            raise ValueError("single-channel DBP (dbp_params 'decim') needs the 'blind' or 'cohmix' receiver")
        self.ref_patmat = _dsp.reference_pattern(np.asarray(sym)[0], np.asarray(sym)[1]) if receiver != 'genie' else None
        self.passes = []
        self.ctx, self.setup, self.sym, self.nsymb, self.nt = ctx, setup, sym, nsymb, nt
        self.nreal, self.batch, self.rank, self.world = nreal, batch, rank, world
        self.r0, self.r1 = shard(nreal, rank, world)
        self.dev = torch.device('cuda', ctx.device)
        self.local = torch.zeros(max(self.r1 - self.r0, 0), dtype=torch.int64, device=self.dev)
        self.tx = _lib.DeviceField(ctx, setup.nfft, setup.nfc, 1)
        self.tx.upload(tx_x, tx_y)
        self.link = Link(ctx, setup, nspan, batch, gain_db, nf_db, self.r0)
        # The genie receiver works in place on the link's stream.  The reference's receive chain is mostly one warp per
        # realization (the adaptive filter is sequential in the symbol index) and leaves the GPU idle: it runs on a context
        # -- a stream -- of its own, in a host thread, beside the propagation of the NEXT group; two work fields alternate.
        self.pipelined = pipeline and receiver != 'genie'
        nslot = 2 if self.pipelined else 1
        self.works = [_lib.DeviceField(ctx, setup.nfft, setup.nfc, batch) for _ in range(nslot)]
        self.bufs = [torch.zeros(batch, dtype=torch.int64, device=self.dev) for _ in range(nslot)]
        self.work, self.buf = self.works[0], self.bufs[0]
        self.rx = None
        self.dbp_genie = None
        if compensation == 'dbp_pmd' and receiver == 'genie':
            from .dbp import dbp_plan
            self.dbp_genie = dbp_plan(ctx, setup, nspan, gain_db, batch=batch, precision='f64', plates=self._link_plates(),
                                      **dict(dbp_params or {}))
        if receiver != 'genie':
            self.rxctx = _lib.Context(ctx.device) if self.pipelined else ctx
            S = None
            if receiver == 'cohmix':
                from . import receiver as _rx
                from .gstate import GSTATE
                x = dict(rx_params or {'oftype': 'gauss', 'obw': 1.9, 'eftype': 'bessel5', 'ebw': 0.65})   # ex20_coherent_polmux.m:47-50
                S = _rx.CohmixSetup(ich, x, GSTATE, nfc=setup.nfc)
            if compensation in ('dbp', 'dbp_pmd'):
                from .dbp import dbp_plan
                dp = dict(dbp_params or {})
                if dp.get('decim') is not None:      # single-channel DBP of the receiver's channel
                    dp['shift'] = S.ndfn if S is not None else 0
                comp = dbp_plan(self.rxctx, setup, nspan, gain_db, batch=batch, precision='f64',
                                plates=self._link_plates() if compensation == 'dbp_pmd' else None, **dp)
            else:
                comp = self.link.cd_plan(self.rxctx)
            self.rx = dict(cd=comp, S=None)
            if receiver == 'cohmix':
                delay = _rx.evaldelay(x['oftype'], x['obw'] * 0.5) + _rx.evaldelay(x['eftype'], x['ebw']) + S.x['post_delay']
                self.rx.update(S=S, ich=ich, shift=int(round(delay * nt)),
                               peak=4.0 * math.sqrt(float(np.asarray(GSTATE.POWER).ravel()[ich - 1])),
                               fo=_lib.Filter(self.rxctx, setup.nfft, 1, S.hf_opt, batch=batch),
                               fe=_lib.Filter(self.rxctx, setup.nfft, 1, _rx.hermitian_part(S.hf_el), batch=batch),
                               col=_lib.DeviceField(self.rxctx, setup.nfft, 1, batch) if setup.nfc > 1 else None)

    def _link_plates(self):
        """the current group's plates as DbpPlan.set_plates takes them: (db0, theta, epsilon), each [nspan][batch][nplates]"""
        return tuple(np.stack([pl[i] for pl in self.link.plates]) for i in range(3))

    def _receive(self, work, buf, g0, nb):
        """the receive chain of one propagated group, on the receiver's context; -> the group's counts land in self.local"""
        from . import dsp as _dsp
        R, c = self.rx, self.rxctx
        R['cd'].execute(work)
        cur, extra = work, {}
        if self.receiver == 'cohmix':
            S = R['S']
            if R['col'] is not None:                                # the channel's column of every realization
                cur = R['col']
                for b in range(self.batch):
                    _lib.field_copy_cols(cur, b, work, b * self.setup.nfc + S.nch - 1, 1)
            if S.ndfn:
                _lib.field_modulate(c, cur, S.ndfn)
            R['fo'].execute(cur)
            _lib.cohmix_exec(c, cur, S.ecw, S.detune, S.lophase, S.balanced)
            R['fe'].execute(cur)
            extra = dict(sample_shift=R['shift'], peak=R['peak'])
        extra.update(self.dsp_params)
        if extra.pop('adcbits', None):                              # p.applyadc (dsp4cohdec.m:157-162)
            _lib.field_quantize(c, cur, int(self.dsp_params['adcbits']))
        passes = _dsp.dsp_count(c, cur, self.nsymb, self.nt, self.ref_patmat, buf.data_ptr(), **extra)   # (synchronises)
        self.local[g0 - self.r0:g0 - self.r0 + nb] = buf[:nb]
        return passes

    def run(self, ase_seed: int = 1):
        """-> (counts [nreal] int64 on the host, Sa*steps done by this rank)"""
        import torch
        sa_steps = 0
        self.local.zero_()
        pool, pending = None, None
        if self.pipelined:
            from concurrent.futures import ThreadPoolExecutor
            pool = ThreadPoolExecutor(max_workers=1)
        try:
            for gi, g0 in enumerate(range(self.r0, self.r1, self.batch)):
                nb = min(self.batch, self.r1 - g0)
                work, buf = self.works[gi % len(self.works)], self.bufs[gi % len(self.bufs)]
                if self.receiver == 'genie':
                    torch.cuda.synchronize(self.dev)                 # torch's stream and the library's are independent
                self.link.retarget(g0)
                work.broadcast_from(self.tx)
                sa_steps += self.link.run(work, ase_seed)            # (returns when the group is propagated)
                if self.receiver == 'genie':
                    if self.dbp_genie is not None:
                        self.dbp_genie.set_plates(*self._link_plates(), plate_sets=self.batch)
                        self.dbp_genie.execute(work)
                    else:
                        self.link.equalize(work)
                    _lib.qpsk_count(self.ctx, work, self.sym, self.nsymb, self.nt, buf.data_ptr())   # writes the send buffer
                    self.ctx.sync()
                    self.local[g0 - self.r0:g0 - self.r0 + nb] = buf[:nb]
                elif pool is None:
                    self._set_rx_plates()
                    self.passes.append(self._receive(work, buf, g0, nb))
                else:
                    if pending is not None:                          # the other slot's receive chain ran beside this link
                        self.passes.append(pending.result())
                    self._set_rx_plates()                            # (before the next retarget draws new plates)
                    pending = pool.submit(self._receive, work, buf, g0, nb)
            if pending is not None:
                self.passes.append(pending.result())
        finally:
            if pool is not None:
                pool.shutdown(wait=True)
        torch.cuda.synchronize(self.dev)
        counts = allreduce_counts(self.local, self.r0, self.nreal)
        return counts.cpu().numpy(), sa_steps

    def _set_rx_plates(self):
        """PMD-aware DBP in the receive chain: this group's plates, while no chain uses the plan"""
        c = self.rx['cd']
        if isinstance(c, _lib.DbpPlan) and c.dbp.pmd:
            c.set_plates(*self._link_plates(), plate_sets=self.batch)

    def close(self):
        if self.dbp_genie is not None:
            self.dbp_genie.close()
        for f in self.works + [self.tx]:
            f.close()
        if self.rx:
            for k in ('fo', 'fe', 'col'):
                if self.rx.get(k) is not None:
                    self.rx[k].close()
            if self.pipelined or isinstance(self.rx['cd'], _lib.DbpPlan):
                self.rx['cd'].close()


def run_mc(ctx: _lib.Context, setup: FiberSetup, tx_x, tx_y, sym, nsymb: int, nt: int, nspan: int, gain_db: float,
           nf_db: float, nreal: int, batch: int, rank: int = 0, world: int = 1, ase_seed: int = 1):
    """One-shot form of McRunner.  -> (counts [nreal] int64 on the host, Sa*steps done by this rank)"""
    r = McRunner(ctx, setup, tx_x, tx_y, sym, nsymb, nt, nspan, gain_db, nf_db, nreal, batch, rank, world)
    try:
        return r.run(ase_seed)
    finally:
        r.close()


def run_mc_native(setup: FiberSetup, tx_x, tx_y, sym, nsymb: int, nt: int, nspan: int, gain_db: float, nf_db: float,
                  nreal: int, batch: int, devices=(0,), ase_seed: int = 1, equalize: bool = True, receiver=None,
                  dsp_params=None, ich: int = 1, dbp_params=None):
    """The same Monte-Carlo job through pmx_mc_run: one process, one host thread and one context per GPU of `devices`,
    the integer all-reduce done with NCCL inside the library (no torch.distributed).  Plate draws as run_mc's.
    receiver: None -- the data-aided counter (with `equalize`); a dict = the x struct of receiver_cohmix -- the reference's
    receive chain (front-end, sampler, DSP core with dsp_params) behind the link, its optical response carrying the
    compensation of the link's chromatic dispersion (as x.dpost / p.applydcf would), or with dbp_params (a dict as
    McRunner's) the digital backpropagation of the link ahead of the front-end and the optical filter alone.
    dbp_params with 'pmd': True -- PMD-aware DBP through every group's own plates: with a receive chain in its place,
    without one (receiver None) in place of the linear equaliser ahead of the data-aided counter; without 'pmd' and
    without a receive chain, dbp_params is ignored.
    -> (counts [nreal] int64, Sa*steps over all realizations)"""
    import ctypes as C
    if dict(dbp_params or {}).get('filter_bw') is not None:
        raise ValueError("run_mc_native: filtered DBP (dbp_params 'filter_bw') is not available in pmx_mc_run; use McRunner")
    if _lib.check_taps(dict(dbp_params or {}).get('nl_taps')).size:
        raise ValueError("run_mc_native: enhanced split-step DBP (dbp_params 'nl_taps') is not available in pmx_mc_run; "
                         "use McRunner")
    lib = _lib.load()
    np_ = setup.nplates
    pl = np.empty((3, nspan, nreal, np_))
    for k in range(nspan):
        for r in range(nreal):
            d = draw_plates(plate_seed(r, k), np_)
            for i in range(3):
                pl[i, k, r] = d[i]
    desc, keep = setup_to_desc(setup, batch=1)
    gain = 10 ** (gain_db * 0.1)
    sigma = np.ascontiguousarray(ase_sigma(gain, nf_db, setup.nfc), dtype=np.float64)
    devs = (C.c_int32 * len(devices))(*[int(d) for d in devices])
    symb = np.ascontiguousarray(sym, dtype=np.uint8).reshape(2, nsymb)
    m = _lib.McDesc()
    m.ndev, m.device_ids, m.nreal, m.batch, m.nspan, m.equalize = len(devices), devs, int(nreal), int(batch), int(nspan), int(equalize)
    m.db0, m.theta, m.epsilon = (pl[i].ctypes.data_as(_lib._dp) for i in range(3))
    m.gain, m.sigma, m.ase_seed = gain, sigma.ctypes.data_as(_lib._dp), int(ase_seed)
    m.sym, m.nsymb, m.nt = symb.ctypes.data_as(C.POINTER(C.c_uint8)), int(nsymb), int(nt)
    rxkeep = None
    dbp_pmd = bool(dict(dbp_params or {}).get('pmd', False))

    def _dbp_desc():
        pd = dict(dbp_params)
        pmd = bool(pd.pop('pmd', False))
        if pd.get('step_len') is None and pd.get('steps_per_span') is None:
            pd['steps_per_span'] = 1
        return _lib.make_dbp(nspan, gain, pmd=pmd, **pd)
    if receiver is None and dbp_pmd:
        dd, dkeep = _dbp_desc()
        m.dbp = C.pointer(dd)
        rxkeep = (dd, dkeep)
    if receiver is not None:
        from . import dsp as _dsp
        from . import receiver as _rx
        from .gstate import GSTATE
        S = _rx.CohmixSetup(ich, receiver, GSTATE, nfc=setup.nfc)
        x = S.x
        delay = _rx.evaldelay(x['oftype'], x['obw'] * 0.5) + _rx.evaldelay(x['eftype'], x['ebw']) + x['post_delay']
        p = dict(dsp_params or {})
        p.update(sample_shift=int(round(delay * nt)), peak=4.0 * math.sqrt(float(np.asarray(GSTATE.POWER).ravel()[ich - 1])))
        if dbp_params is None:
            ph = np.asarray(setup.betat, dtype=np.float64)[:, 0] * (setup.length * nspan)      # the link's all-pass phase, undone
            hopt = np.ascontiguousarray(S.hf_opt * (np.cos(ph) + 1j * np.sin(ph)))
        else:
            hopt = np.ascontiguousarray(np.asarray(S.hf_opt, dtype=np.complex128))
        hel = np.ascontiguousarray(np.asarray(S.hf_el, dtype=np.complex128))
        ref = np.ascontiguousarray(_dsp.reference_pattern(np.asarray(sym)[0], np.asarray(sym)[1]), dtype=np.uint8)
        lop = None if S.lophase is None else np.ascontiguousarray(S.lophase, dtype=np.float64)
        rx = _lib.McReceiver()
        rx.hf_opt, rx.hf_el = hopt.ctypes.data_as(_lib._dp), hel.ctypes.data_as(_lib._dp)
        rx.lo_ecw, rx.lo_detune, rx.balanced = float(S.ecw), float(S.detune), int(S.balanced)
        rx.lo_phase = None if lop is None else lop.ctypes.data_as(_lib._dp)
        rx.dsp = _dsp._desc(nsymb, nt, p)
        rx.ref_patmat = ref.ctypes.data_as(C.POINTER(C.c_uint8))
        if dbp_params is not None:
            dd, dkeep = _dbp_desc()
            rx.dbp = C.pointer(dd)
            rxkeep = (hopt, hel, ref, lop, rx, dd, dkeep)
        else:
            rxkeep = (hopt, hel, ref, lop, rx)
        m.rx = C.pointer(rx)
        m.equalize = 0
    fx = np.ascontiguousarray(np.asarray(tx_x, dtype=np.complex128).T)[None]
    fy = np.ascontiguousarray(np.asarray(tx_y, dtype=np.complex128).T)[None]
    io = _lib.complex_field(fx, fy)
    counts = np.zeros(nreal, dtype=np.int64)
    sa = C.c_int64(0)
    err = C.create_string_buffer(512)
    rc = lib.pmx_mc_run(C.byref(desc), C.byref(m), C.byref(io), counts.ctypes.data_as(C.POINTER(C.c_int64)), C.byref(sa), err, 512)
    if rc != 0:
        raise _lib.PolmuxError(rc, err.value.decode(errors='replace'))
    return counts, int(sa.value)
