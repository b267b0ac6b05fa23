"""-m gpu: forward-path kernel instances at the edges of their inputs.

* The full-angle nonlinear step.  pmx_ctl_next flags a step PMX_BM_NL_SMALL when its largest nonlinear phase
  gam*leff*max|u|^2 is below 2^-6; passes A and C and the on-chip kernel then take the Taylor kernel pmx_cis_small
  instead of the reduced sine / cosine pmx_cis_r.  Fibres at the reference's dphimax of a few mrad never leave the Taylor
  branch.  Here the step is bounded by the nonlinear phase (firstdz < dzmax: the first step's phase is dphimax itself)
  at 2^-6 (on the threshold), 0.02, 1 rad and 3 rad; at 3 rad the CNLSE rotation angle (up to a third of the phase,
  1 rad) passes pi/4, so pmx_cis_r's other quadrants run.  FP64 <= 1e-10 against the oracle, step counts and trunk
  schedules equal; FP32 <= 1e-5.
* A batch whose realization groups hold more than PMX_LIVE_CAP = 64 realizations: the passes then read the done-flags
  from the step packages in global memory instead of their per-CTA cache.
* The limit of batch*nfc <= 65535 realization-columns (the kernels put them in gridDim.y): refused up front, and run
  at the limit."""
import numpy as np
import pytest

import oracle.fiber_oracle as orc
import polmux_b200 as pmx
from polmux_b200 import _lib, mc
from polmux_b200.fiber import fiber_setup, setup_to_desc
from common import base_fiber, make_tx, rel_l2

pytestmark = pytest.mark.gpu
TOL = 1e-10
TOL32 = 1e-5

LEVELS = [2.0 ** -6, 0.02, 1.0, 3.0]                            # nonlinear phase of a step, rad
NL_CASES = [('gps-', 'yes'), ('gps-', 'no'), ('g-s-', 'no')]   # Manakov, CNLSE with plates, CNLSE without plates


def _full_angle_fiber(level, flag, manakov, leff=1e3, dzmax=2e4, length=None):
    """A fibre whose first step is bounded by the nonlinear phase `level` at leff (the step's effective length): n2 scaled
    so that gam*leff*max|u|^2 = level for the field in GSTATE.  6 km, or 3 km from 1 rad per step up: a propagation of
    tens of radians of nonlinear phase amplifies a relative perturbation of 1e-13 of the input to 1e-10 and more (the
    oracle's own sensitivity), and the parity bar would measure that instead of the kernels."""
    G = pmx.GSTATE
    pmax = float(np.max(np.abs(G.FIELDX) ** 2 + np.abs(G.FIELDY) ** 2))
    if length is None:
        length = 6e3 if level < 0.1 else 3e3
    fib = base_fiber(length=length, dzmax=dzmax, dphimax=level, manakov=manakov)
    if 'p' in flag:
        fib.update(dgd=0.3, nplates=4)
    gam = fiber_setup(fib, flag, rng=np.random.Generator(np.random.PCG64(0))).gam[0]
    fib['n2'] = fib['n2'] * level / (leff * gam * pmax)
    return fib


def _schedule_equal(L, log):
    assert L['ncycle'] == log['ncycle']
    assert list(L['trace_ntrunk'])[:L['ncycle']] == [s['ntrunk'] for s in log['schedule']]
    np.testing.assert_allclose(list(L['trace_dz'])[:L['ncycle']], [s['dz'] for s in log['schedule']], rtol=1e-9)
    np.testing.assert_allclose(L['firstdz'], log['firstdz'], rtol=1e-13)


@pytest.mark.parametrize('level', LEVELS)
@pytest.mark.parametrize('flag,manakov', NL_CASES)
@pytest.mark.parametrize('lg', [10, 14])
def test_full_angle_nonlinear_step_against_oracle(lg, flag, manakov, level):
    """2^10: the on-chip kernel; 2^14: the three passes with a batch of one (step control fused into pass A)"""
    gs = make_tx((1 << lg) // 16, 16)
    fib = _full_angle_fiber(level, flag, manakov)
    orc.fiber(gs, fib, flag, rng=np.random.Generator(np.random.PCG64(5)))
    pmx.fiber(fib, flag, rng=np.random.Generator(np.random.PCG64(5)), trace=True)
    G, L = pmx.GSTATE, pmx.FIBER_LAST
    _schedule_equal(L, gs.log)
    assert gs.log['firstdz'] < fib['dzmax'] and gs.log['ncycle'] >= 4
    err = rel_l2(G.FIELDX, G.FIELDY, gs.FIELDX, gs.FIELDY)
    print('full-angle FP64 lg=%d %s manakov=%s phase=%.4g rad: rel-L2 %.3e, %d steps' % (lg, flag, manakov, level, err,
                                                                                     L['ncycle']))
    assert err < TOL


@pytest.mark.parametrize('level', LEVELS)
@pytest.mark.parametrize('flag,manakov', NL_CASES)
def test_full_angle_nonlinear_step_batch_of_three(flag, manakov, level):
    """three realizations at 2^14 (the step-control kernel pmx_k_ctl between the passes), powers 1, 1.05^2, 1.1^2: each
    against its own oracle run"""
    nsymb, nt, batch = 1 << 10, 16, 3
    n = nsymb * nt
    make_tx(nsymb, nt)
    G = pmx.GSTATE
    x0, y0 = np.array(G.FIELDX), np.array(G.FIELDY)
    fib = _full_angle_fiber(level, flag, manakov)
    setup = fiber_setup(fib, flag, rng=np.random.Generator(np.random.PCG64(6)))
    ctx = _lib.default_context()
    scale = [1.0 + 0.05 * b for b in range(batch)]
    work = _lib.DeviceField(ctx, n, 1, batch)
    work.upload(np.stack([s * x0.T for s in scale]), np.stack([s * y0.T for s in scale]))
    desc, keep = setup_to_desc(setup, batch=batch)
    plan = _lib.Plan(ctx, desc, keep)
    res = plan.execute(work, trace_cap=4096)
    gx, gy = work.download()
    plan.close()
    work.close()
    for b in range(batch):
        gs = make_tx(nsymb, nt)
        gs.FIELDX, gs.FIELDY = gs.FIELDX * scale[b], gs.FIELDY * scale[b]
        orc.fiber(gs, fib, flag, rng=np.random.Generator(np.random.PCG64(6)))
        dz, ntr = res.schedule(b)
        _schedule_equal(dict(ncycle=int(res.ncycle[b]), trace_dz=dz, trace_ntrunk=ntr, firstdz=res.firstdz[b]), gs.log)
        assert gs.log['firstdz'] < fib['dzmax']
        err = rel_l2(gx[b].T, gy[b].T, gs.FIELDX, gs.FIELDY)
        print('full-angle FP64 batch 3, b=%d %s manakov=%s phase=%.4g rad: rel-L2 %.3e' % (b, flag, manakov, level, err))
        assert err < TOL, (b, err)


@pytest.mark.parametrize('lg', [10, 14])
def test_full_angle_step_capped_by_dzmax(lg):
    """steps of 1 km bounded by dzmax, where the phase bound would allow 3 km: about 1/3 rad, the general kernel"""
    gs = make_tx((1 << lg) // 16, 16)
    fib = _full_angle_fiber(1.0, 'gps-', 'no', leff=3e3, dzmax=1e3, length=6e3)
    orc.fiber(gs, fib, 'gps-', rng=np.random.Generator(np.random.PCG64(8)))
    pmx.fiber(fib, 'gps-', rng=np.random.Generator(np.random.PCG64(8)), trace=True)
    G, L = pmx.GSTATE, pmx.FIBER_LAST
    _schedule_equal(L, gs.log)
    assert gs.log['firstdz'] == fib['dzmax']
    assert rel_l2(G.FIELDX, G.FIELDY, gs.FIELDX, gs.FIELDY) < TOL


@pytest.mark.parametrize('flag,manakov', [('gps-', 'no'), ('g-s-', 'no')])
@pytest.mark.parametrize('lg', [10, 14])
def test_fp32_full_angle_nonlinear_step(lg, flag, manakov):
    """FP32 at 1 rad per step (pmx_cis_r in float, CNLSE rotation): <= 1e-5 against the FP64 oracle, ncycle within one.
    2 km (three steps): FP32's rounding grows by about 2e-7 per step, and more at full angles, where the propagation
    amplifies it (3 km, 6 km: 2e-5 and more)"""
    gs = make_tx((1 << lg) // 16, 16)
    fib = _full_angle_fiber(1.0, flag, manakov, length=2e3)
    orc.fiber(gs, fib, flag, rng=np.random.Generator(np.random.PCG64(9)))
    pmx.fiber(fib, flag, rng=np.random.Generator(np.random.PCG64(9)), precision='f32')
    G = pmx.GSTATE
    err = rel_l2(G.FIELDX, G.FIELDY, gs.FIELDX, gs.FIELDY)
    print('full-angle FP32 lg=%d %s phase=1 rad: rel-L2 %.3e, %d steps' % (lg, flag, err, pmx.FIBER_LAST['ncycle']))
    assert gs.log['firstdz'] < fib['dzmax']
    assert abs(pmx.FIBER_LAST['ncycle'] - gs.log['ncycle']) <= 1
    assert err < TOL32


def test_ragged_batch_above_the_done_flag_cache():
    """150 realizations at 2^13 (three passes, 64 x 128), each with its own plate draw and power.  The batch is split into
    two realization groups of 75 on two streams (plan_groups: 32 tiles per realization for pass A, 4800 tiles > two
    rounds of 148 SMs x 16 resident CTAs), so every pass sees more than PMX_LIVE_CAP = 64 realizations and reads their
    done-flags from global memory.  The realizations at group index 64 and above run at the lowest power and finish
    first: the passes must skip them from then on.  Every realization equals its own single run bit for bit."""
    nsymb, nt, batch, ngroup = 512, 16, 150, 75
    n = nsymb * nt
    make_tx(nsymb, nt)
    G = pmx.GSTATE
    fib = base_fiber(length=3e4, dgd=0.4, nplates=6, manakov='yes')
    setup = fiber_setup(fib, 'gps-', rng=np.random.Generator(np.random.PCG64(0)))
    draws = [mc.draw_plates(mc.plate_seed(b, 0), setup.nplates) for b in range(batch)]
    pl = [np.stack([d[i] for d in draws]) for i in range(3)]
    scale = [0.6 if b % ngroup >= 64 else 1.0 + 0.1 * (b % 4) for b in range(batch)]
    ctx = _lib.default_context()
    x0 = np.stack([np.ascontiguousarray((G.FIELDX * s).T) for s in scale])
    y0 = np.stack([np.ascontiguousarray((G.FIELDY * s).T) for s in scale])
    work = _lib.DeviceField(ctx, n, 1, batch)
    work.upload(x0, y0)
    desc, keep = setup_to_desc(setup, batch=batch, plate_sets=batch, db0=pl[0], theta=pl[1], epsilon=pl[2])
    plan = _lib.Plan(ctx, desc, keep)
    res = plan.execute(work)
    gx, gy = work.download()
    plan.close()
    late = [b for b in range(batch) if b % ngroup >= 64]
    assert max(int(res.ncycle[b]) for b in late) < int(res.ncycle.max())     # they finish while others still run
    assert len(set(int(v) for v in res.ncycle)) > 1
    one = _lib.DeviceField(ctx, n, 1, 1)
    for b in range(batch):
        one.upload(x0[b:b + 1], y0[b:b + 1])
        d1, k1 = setup_to_desc(setup, batch=1, plate_sets=1, db0=pl[0][b][None], theta=pl[1][b][None], epsilon=pl[2][b][None])
        p1 = _lib.Plan(ctx, d1, k1)
        r1 = p1.execute(one)
        ox, oy = one.download()
        p1.close()
        assert int(r1.ncycle[0]) == int(res.ncycle[b]), b
        assert np.array_equal(ox[0], gx[b]) and np.array_equal(oy[0], gy[b]), b
    for f in (work, one):
        f.close()


def test_batch_times_columns_above_65535_is_refused():
    """a field or a plan of more than 65535 realization-columns: PolmuxError naming the limit, and nothing launched"""
    ctx = _lib.default_context()
    make_tx(4, 16)
    setup = fiber_setup(base_fiber(length=1e3, dgd=0.1, nplates=2, manakov='yes'), 'gps-',
                        rng=np.random.Generator(np.random.PCG64(0)))
    before = ctx.launches
    for nfc, batch in ((1, 65536), (2, 32768), (8, 8192)):
        with pytest.raises(_lib.PolmuxError, match='65535'):
            _lib.DeviceField(ctx, 64, nfc, batch)
    desc, keep = setup_to_desc(setup, batch=65536)
    with pytest.raises(_lib.PolmuxError, match='65535'):
        _lib.Plan(ctx, desc, keep)
    with pytest.raises(_lib.PolmuxError, match='65535'):
        _lib.Filter(ctx, 1 << 12, 2, np.ones(1 << 12), batch=32768)
    dbp, dkeep = _lib.make_dbp(1, steps_per_span=2)
    desc, keep = setup_to_desc(setup, batch=65536)
    with pytest.raises(_lib.PolmuxError, match='65535'):
        _lib.DbpPlan(ctx, desc, keep, dbp, dkeep)
    assert ctx.launches == before


def test_batch_of_65535_small_realizations():
    """65535 realizations of 2^6 samples (the largest batch of one column): fiber on the on-chip kernel, then ampliflat
    with injected noise.  The first, the last and three middle realizations equal their single fiber runs bit for bit,
    and ampliflat equals u*sqrt(G) + sigma*noise in numpy."""
    nsymb, nt, batch = 4, 16, 65535
    n = nsymb * nt
    make_tx(nsymb, nt)
    G = pmx.GSTATE
    fib = base_fiber(length=2e4, dgd=0.3, nplates=5, manakov='no')
    setup = fiber_setup(fib, 'gps-', rng=np.random.Generator(np.random.PCG64(1)))
    ctx = _lib.default_context()
    scale = 1.0 + 0.5 * (np.arange(batch) % 7) / 7
    x0 = np.asarray(G.FIELDX).T[None] * scale[:, None, None]
    y0 = np.asarray(G.FIELDY).T[None] * scale[:, None, None]
    work = _lib.DeviceField(ctx, n, 1, batch)
    work.upload(x0, y0)
    desc, keep = setup_to_desc(setup, batch=batch)
    plan = _lib.Plan(ctx, desc, keep)
    res = plan.execute(work)
    plan.close()
    picks = [0, 21845, 32767, 43690, batch - 1]
    mid = {b: work.download(b, 1) for b in picks}
    one = _lib.DeviceField(ctx, n, 1, 1)
    d1, k1 = setup_to_desc(setup, batch=1)
    p1 = _lib.Plan(ctx, d1, k1)
    for b in picks:
        one.upload(x0[b:b + 1], y0[b:b + 1])
        r1 = p1.execute(one)
        ox, oy = one.download()
        assert int(r1.ncycle[0]) == int(res.ncycle[b]), b
        assert np.array_equal(ox, mid[b][0]) and np.array_equal(oy, mid[b][1]), b
    p1.close()
    one.close()
    assert len(set(int(res.ncycle[b]) for b in picks)) > 1
    gain, sigma = 4.0, 0.25
    noise = np.random.Generator(np.random.PCG64(2)).standard_normal((batch, 2, n, 2)).view(np.complex128)[..., 0]
    _lib.ampliflat_exec(ctx, work, gain, [sigma], noise=noise)
    for b in picks:
        gx, gy = work.download(b, 1)
        rx = mid[b][0][0, 0] * np.sqrt(gain) + sigma * noise[b, 0]
        ry = mid[b][1][0, 0] * np.sqrt(gain) + sigma * noise[b, 1]
        assert rel_l2(gx[0, 0], gy[0, 0], rx, ry) < 1e-14, b
    work.close()
