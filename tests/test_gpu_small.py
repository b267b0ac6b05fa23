"""-m gpu: small fields (2^6 ... 2^12 samples per column) -- the single-launch on-chip kernel (pmx_onchip.cuh: one CTA
per realization-column, the whole matrix_ssfm / scalar_ssfm loop in shared memory and registers, the columns of a
realization in one thread-block cluster) against the oracle, at the sizes of the reference's own scalar-path scripts
(ex06_ber.m:14-16: 2^10, ex10_wdm.m:22-24: 2^11 x 5 channels with XPM) and below; at 2^12 also against the three-pass
kernels (PMX_NO_ONCHIP=1).  FP64 <= 1e-10, step counts and trunk schedules equal."""
import os

import numpy as np
import pytest

import oracle.fiber_oracle as orc
import polmux_b200 as pmx
from polmux_b200 import _lib, mc
from polmux_b200.fiber import fiber_setup, setup_to_desc
from common import base_fiber, make_tx, rel_l2, scalar_tx as _scalar_tx

pytestmark = pytest.mark.gpu
TOL = 1e-10


def _check(gs, fib, flag, seed=7, two_pol=True, disp_mode=None):
    orc.fiber(gs, fib, flag, rng=np.random.Generator(np.random.PCG64(seed)))
    pmx.fiber(fib, flag, rng=np.random.Generator(np.random.PCG64(seed)), trace=two_pol, disp_mode=disp_mode)
    G, L = pmx.GSTATE, pmx.FIBER_LAST
    assert L['ncycle'] == gs.log['ncycle']
    if two_pol:
        assert list(L['trace_ntrunk'])[:L['ncycle']] == [s['ntrunk'] for s in gs.log['schedule']]
        return rel_l2(G.FIELDX, G.FIELDY, gs.FIELDX, gs.FIELDY)
    return float(np.linalg.norm(G.FIELDX - gs.FIELDX) / np.linalg.norm(gs.FIELDX))


@pytest.mark.parametrize('manakov', ['yes', 'no'])
@pytest.mark.parametrize('lg', [6, 7, 8, 9, 10, 11, 12])
def test_two_pol_pmd_every_small_size(lg, manakov):
    """'gps-' with PMD plates at every on-chip transform length 64 ... 4096"""
    nt = 8 if lg < 9 else 16
    gs = make_tx((1 << lg) // nt, nt)
    fib = base_fiber(length=5e4, dgd=0.4, nplates=12, manakov=manakov)
    assert _check(gs, fib, 'gps-') < TOL


@pytest.mark.parametrize('manakov', ['yes', 'no'])
@pytest.mark.parametrize('lg', [6, 7, 8, 9, 10, 11])
def test_two_pol_pmd_every_small_size_vector_dispersion(lg, manakov):
    """the same in vector dispersion mode (betat / db1 uploaded, pmx_k_onchip<..., SC = false>)"""
    nt = 8 if lg < 9 else 16
    gs = make_tx((1 << lg) // nt, nt)
    fib = base_fiber(length=5e4, dgd=0.4, nplates=12, manakov=manakov)
    assert _check(gs, fib, 'gps-', disp_mode='vector') < TOL


@pytest.mark.parametrize('nch,lg', [(3, 10), (8, 9)])
def test_sepfields_in_one_cluster_vector_dispersion(nch, lg):
    """per-column betat / db1 tables of a cluster in vector dispersion mode"""
    gs = make_tx((1 << lg) // 16, 16, nch=nch, ftype='sepfields', pavg_mw=1.5)
    fib = base_fiber(length=4e4, dgd=0.3, nplates=10, manakov='yes', slope=0.057)
    assert _check(gs, fib, 'gps-', disp_mode='vector') < TOL


@pytest.mark.parametrize('nsymb,nt,nch,flag', [(32, 32, 1, 'g-sx'), (64, 32, 5, 'g-sx')])
def test_scalar_path_vector_dispersion(nsymb, nt, nch, flag):
    gs = _scalar_tx(nsymb, nt, nch)
    fib = base_fiber(length=1e5, dphimax=3e-3, slope=0.057)
    assert _check(gs, fib, flag, two_pol=False, disp_mode='vector') < TOL


@pytest.mark.parametrize('flag', ['g---', 'gp--', '--s-', 'g-s-', '-ps-'])
def test_flags_small(flag):
    gs = make_tx(64, 16)
    fib = base_fiber(length=4e4, dgd=0.3, nplates=20, manakov='no')
    assert _check(gs, fib, flag) < TOL


@pytest.mark.parametrize('nch,lg', [(2, 8), (3, 10), (5, 11), (8, 9)])
def test_sepfields_columns_in_one_cluster(nch, lg):
    """'sepfields' (nfc = nch columns, one CTA each, one cluster per realization): the step control sees the maximum
    over the columns (fiber.m:694-698)"""
    gs = make_tx((1 << lg) // 16, 16, nch=nch, ftype='sepfields', pavg_mw=1.5)
    fib = base_fiber(length=4e4, dgd=0.3, nplates=10, manakov='yes', slope=0.057)
    assert _check(gs, fib, 'gps-') < TOL


@pytest.mark.parametrize('nsymb,nt,nch,flag', [(32, 32, 1, 'g-sx'), (64, 32, 5, 'g-sx'), (64, 32, 5, 'g--x'), (32, 16, 3, 'g-s-'),
                                                (16, 16, 8, 'g-sx')])
def test_scalar_path_with_xpm_over_the_cluster(nsymb, nt, nch, flag):
    """the scalar path at the sizes of ex06_ber.m (32 x 32, one channel) and ex10_wdm.m (64 x 32, five separate
    channels): nl_step's cross-column sum of |u|^2 (fiber.m:793-799) read through distributed shared memory"""
    gs = _scalar_tx(nsymb, nt, nch)
    fib = base_fiber(length=1e5, dphimax=3e-3, slope=0.057)
    assert _check(gs, fib, flag, two_pol=False) < TOL


def test_on_chip_and_three_pass_kernels_agree_at_4096():
    """2^12 samples run on chip by default; PMX_NO_ONCHIP=1 sends them through passes A/B/C (64 x 64 split)"""
    fib = base_fiber(length=6e4, dgd=0.5, nplates=15, manakov='no')
    outs = []
    for env in ('0', '1'):
        os.environ['PMX_NO_ONCHIP'] = env
        try:
            gs = make_tx(256, 16)
            err = _check(gs, fib, 'gps-')
            assert err < TOL
            outs.append((np.array(pmx.GSTATE.FIELDX), np.array(pmx.GSTATE.FIELDY), pmx.FIBER_LAST['ncycle']))
        finally:
            os.environ.pop('PMX_NO_ONCHIP', None)
    assert outs[0][2] == outs[1][2]
    assert rel_l2(outs[0][0], outs[0][1], outs[1][0], outs[1][1]) < 1e-12


def test_batch_of_small_realizations_ragged():
    """a resident batch of small fields with different plate draws and powers (different step counts): every
    realization equals its own single run bit for bit"""
    nsymb, nt, batch = 64, 16, 5
    n = nsymb * nt
    make_tx(nsymb, nt)
    G = pmx.GSTATE
    fib = base_fiber(length=5e4, dgd=0.4, nplates=9, manakov='yes')
    setup = fiber_setup(fib, 'gps-', rng=np.random.Generator(np.random.PCG64(0)))
    draws = [mc.draw_plates(mc.plate_seed(b, 0), setup.nplates) for b in range(batch)]
    pl = [np.stack([d[i] for d in draws]) for i in range(3)]
    ctx = _lib.default_context()
    x0 = np.stack([np.ascontiguousarray((G.FIELDX * (1 + 0.2 * b)).T) for b in range(batch)])
    y0 = np.stack([np.ascontiguousarray((G.FIELDY * (1 + 0.2 * b)).T) for b in range(batch)])
    work = _lib.DeviceField(ctx, n, 1, batch)
    work.upload(x0, y0)
    desc, keep = setup_to_desc(setup, batch=batch, plate_sets=batch, db0=pl[0], theta=pl[1], epsilon=pl[2])
    plan = _lib.Plan(ctx, desc, keep)
    res = plan.execute(work)
    gx, gy = work.download()
    plan.close()
    one = _lib.DeviceField(ctx, n, 1, 1)
    for b in range(batch):
        one.upload(x0[b:b + 1], y0[b:b + 1])
        d1, k1 = setup_to_desc(setup, batch=1, plate_sets=1, db0=pl[0][b][None], theta=pl[1][b][None], epsilon=pl[2][b][None])
        p1 = _lib.Plan(ctx, d1, k1)
        r1 = p1.execute(one)
        ox, oy = one.download()
        p1.close()
        assert int(r1.ncycle[0]) == int(res.ncycle[b])
        assert np.array_equal(ox[0], gx[b]) and np.array_equal(oy[0], gy[b])
    assert len(set(int(v) for v in res.ncycle)) > 1
    for f in (work, one):
        f.close()


def test_small_field_limits():
    """below 2^6 samples, or more than 8 columns below 2^12: PMX_ERR_UNSUPPORTED with a message"""
    gs = make_tx(2, 16)
    with pytest.raises(_lib.PolmuxError, match='2\\^6'):
        pmx.fiber(base_fiber(length=1e4), 'g-s-')
    make_tx(16, 16, nch=9, ftype='sepfields')
    with pytest.raises(_lib.PolmuxError, match='at most 8 columns'):
        pmx.fiber(base_fiber(length=1e4, dgd=0.1, nplates=4, manakov='yes'), 'gps-')
