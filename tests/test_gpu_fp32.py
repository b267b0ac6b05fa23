"""-m gpu: the FP32 mode of the CUDA path (pmx_fiber_desc.precision = PMX_F32) against the FP64 numpy oracle.

BASELINE.json north_star: "an FP32 mode is reported separately with <= 1e-5 tolerance" -- relative L2 error of the
output field against the reference's (FP64) result.  The step schedule is produced by the same device-side
step control from float data, so ncycle may differ by a step where a boundary is hit within float rounding;
it is compared with a tolerance of one step."""
import numpy as np
import pytest

import oracle.fiber_oracle as orc
import polmux_b200 as pmx
from common import base_fiber, make_tx, rel_l2, scalar_tx

pytestmark = pytest.mark.gpu
TOL32 = 1e-5


@pytest.fixture(autouse=True, params=['scalar', 'vector'])
def disp_mode(request, monkeypatch):
    import importlib
    fmod = importlib.import_module('polmux_b200.fiber')
    monkeypatch.setattr(fmod, 'DISP_MODE', request.param)
    return request.param


_ORACLE = {}


def run32(nsymb, nt, fib, flag, nch=1, ftype='unique', seed=1000, pavg=2.0, cache=None):
    """cache: a key under which the oracle's output is kept for the other dispersion mode (long fields)"""
    gs = make_tx(nsymb, nt, nch, ftype=ftype, pavg_mw=pavg)
    if cache is not None and cache in _ORACLE:
        gs.FIELDX, gs.FIELDY, gs.log = _ORACLE[cache]
    else:
        orc.fiber(gs, fib, flag, rng=np.random.Generator(np.random.PCG64(seed)))
        if cache is not None:
            _ORACLE[cache] = (gs.FIELDX, gs.FIELDY, gs.log)
    pmx.fiber(fib, flag, rng=np.random.Generator(np.random.PCG64(seed)), precision='f32')
    G = pmx.GSTATE
    err = rel_l2(G.FIELDX, G.FIELDY, gs.FIELDX, gs.FIELDY)
    print('FP32 %d x %d x %d %s: rel-L2 %.3e, %d steps' % (nsymb, nt, nch, flag, err, pmx.FIBER_LAST['ncycle']))
    return err, gs


def ncycle_within_one(gs):
    return abs(pmx.FIBER_LAST['ncycle'] - gs.log['ncycle']) <= 1


@pytest.mark.parametrize('lg', [12, 14, 16, 18])
def test_fp32_linear_gvd(lg):
    err, gs = run32(1 << (lg - 4), 16, base_fiber(length=1e5), 'g---')
    assert err < TOL32
    assert pmx.FIBER_LAST['ncycle'] == 1


@pytest.mark.parametrize('lg,nplates', [(12, 10), (16, 200)])
def test_fp32_linear_pmd(lg, nplates):
    err, gs = run32(1 << (lg - 4), 16, base_fiber(dgd=0.5, nplates=nplates), 'gp--')
    assert err < TOL32


@pytest.mark.parametrize('lg,manakov', [(14, 'no'), (14, 'yes'), (16, 'yes'), (17, 'no')])
def test_fp32_nonlinear_pmd(lg, manakov):
    """C1-like: 100 km, 'gps-', 10 plates, CNLSE and Manakov (about 45 steps)."""
    fib = base_fiber(length=1e5, dgd=1.0, nplates=10, manakov=manakov)
    err, gs = run32(1 << (lg - 4), 16, fib, 'gps-')
    assert err < TOL32
    assert abs(pmx.FIBER_LAST['ncycle'] - gs.log['ncycle']) <= 1


def test_fp32_sepfields_spm():
    """two 'sepfields' columns, SPM only (no 'p'): per-column gamma."""
    fib = base_fiber(length=5e4)
    err, gs = run32(1 << 10, 16, fib, 'g-s-', nch=2, ftype='sepfields')
    assert err < TOL32


@pytest.mark.parametrize('manakov', ['yes', 'no'])
@pytest.mark.parametrize('lg', [6, 7, 8, 9, 10, 11, 12])
def test_fp32_onchip_nonlinear_pmd(lg, manakov):
    """'gps-' on the on-chip kernel (pmx_k_onchip<float, L>: step control, max reduction) at every length 64 ... 4096"""
    nt = 8 if lg < 9 else 16
    fib = base_fiber(length=5e4, dgd=0.4, nplates=12, manakov=manakov)
    err, gs = run32((1 << lg) // nt, nt, fib, 'gps-')
    assert err < TOL32
    assert ncycle_within_one(gs)


@pytest.mark.parametrize('nch,lg', [(3, 10), (8, 9)])
def test_fp32_sepfields_columns_in_one_cluster(nch, lg):
    """'sepfields' on chip: 3 and 8 columns, one CTA each, the step control's maximum over the cluster"""
    fib = base_fiber(length=4e4, dgd=0.3, nplates=10, manakov='yes', slope=0.057)
    err, gs = run32((1 << lg) // 16, 16, fib, 'gps-', nch=nch, ftype='sepfields')
    assert err < TOL32
    assert ncycle_within_one(gs)


def test_fp32_sepfields_many_columns_three_pass():
    """24 'sepfields' columns at 2^13: the three passes with the realization-column split (nfc_magic)"""
    fib = base_fiber(length=2e4, dgd=0.3, nplates=10, manakov='yes', slope=0.057)
    err, gs = run32(1 << 9, 16, fib, 'gps-', nch=24, ftype='sepfields', pavg=0.5)
    assert err < TOL32
    assert ncycle_within_one(gs)


@pytest.mark.parametrize('lg,no_onchip', [(13, False), (12, True)])
def test_fp32_three_pass_length_64(lg, no_onchip, monkeypatch):
    """the three passes at L = 64: 2^13 (64 x 128) and 2^12 with PMX_NO_ONCHIP=1 (64 x 64)"""
    if no_onchip:
        monkeypatch.setenv('PMX_NO_ONCHIP', '1')
    fib = base_fiber(length=5e4, dgd=0.5, nplates=15, manakov='no')
    err, gs = run32(1 << (lg - 4), 16, fib, 'gps-')
    assert err < TOL32
    assert ncycle_within_one(gs)


@pytest.mark.parametrize('lg,nt,length,nplates,manakov', [
    (22, 64, 4.0e3, 4, 'yes'),     # 2048 x 2048: passes A, B and C at L = 2048
    (24, 64, 3.0e3, 3, 'no'),      # 4096 x 4096: L = 4096, CNLSE
])
def test_fp32_gps_prefix_long_transforms(lg, nt, length, nplates, manakov):
    """the L = 2048 and L = 4096 pass instances (2^21 and 2^23 run the same kernels as 2^22 and 2^24) on a short 'gps-'
    prefix with whole and partial trunks; the oracle (seconds per trunk here) runs once for both dispersion modes"""
    fib = base_fiber(length=length, dgd=0.3, nplates=nplates, manakov=manakov)
    err, gs = run32((1 << lg) // nt, nt, fib, 'gps-', seed=1000 + lg, cache=lg)
    sched = gs.log['schedule']
    assert gs.log['ncycle'] >= 3 and sum(s['ntrunk'] for s in sched) > gs.log['ncycle']
    assert err < TOL32
    assert ncycle_within_one(gs)


@pytest.mark.parametrize('nsymb,nt,nch,flag', [(32, 32, 1, 'g-sx'), (64, 32, 5, 'g-sx'), (64, 32, 5, 'g--x'),
                                                (64, 32, 5, 'g-s-'), (256, 32, 3, 'g-sx')])
def test_fp32_scalar_path(nsymb, nt, nch, flag):
    """the scalar path in FP32 at the shapes of ex06_ber.m (32 x 32) and ex10_wdm.m (64 x 32, five channels) on chip, and
    three columns with 'x' at 2^13 on the three passes (pmx_k_xpm_sum<float>, pass A clearing the Y slot)"""
    gs = scalar_tx(nsymb, nt, nch)
    fib = base_fiber(length=3e4, dphimax=5e-3, slope=0.057)     # about 35 steps
    orc.fiber(gs, fib, flag)
    pmx.fiber(fib, flag, precision='f32')
    G = pmx.GSTATE
    err = float(np.linalg.norm(G.FIELDX - gs.FIELDX) / np.linalg.norm(gs.FIELDX))
    print('FP32 scalar %d x %d x %d %s: rel-L2 %.3e, %d steps' % (nsymb, nt, nch, flag, err, pmx.FIBER_LAST['ncycle']))
    assert err < TOL32
    assert ncycle_within_one(gs)


def test_fp32_batch_ragged_three_pass():
    """an FP32 resident batch at 2^13 (three passes) with different plate draws and powers: every realization equals its
    own single run bit for bit, and the finished realizations are skipped"""
    from polmux_b200 import _lib, mc
    from polmux_b200.fiber import fiber_setup, setup_to_desc
    nsymb, nt, batch = 512, 16, 5
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
    work = _lib.DeviceField(ctx, n, 1, batch, precision=_lib.PMX_F32)
    work.upload(x0, y0)
    desc, keep = setup_to_desc(setup, batch=batch, plate_sets=batch, db0=pl[0], theta=pl[1], epsilon=pl[2], precision='f32')
    plan = _lib.Plan(ctx, desc, keep)
    res = plan.execute(work)
    gx, gy = work.download()
    plan.close()
    one = _lib.DeviceField(ctx, n, 1, 1, precision=_lib.PMX_F32)
    for b in range(batch):
        one.upload(x0[b:b + 1], y0[b:b + 1])
        d1, k1 = setup_to_desc(setup, batch=1, plate_sets=1, db0=pl[0][b][None], theta=pl[1][b][None], epsilon=pl[2][b][None],
                               precision='f32')
        p1 = _lib.Plan(ctx, d1, k1)
        r1 = p1.execute(one)
        ox, oy = one.download()
        p1.close()
        assert int(r1.ncycle[0]) == int(res.ncycle[b])
        assert np.array_equal(ox[0], gx[b]) and np.array_equal(oy[0], gy[b])
    assert len(set(int(v) for v in res.ncycle)) > 1
    for f in (work, one):
        f.close()


def test_fp32_ampliflat_gain_and_injected_noise():
    """ampliflat on an FP32 field: u*sqrt(G) + sigma*noise (ampliflat.m:78-148) against numpy, float rounding only."""
    from polmux_b200 import _lib
    ctx = _lib.default_context()
    n = 1 << 12
    rng = np.random.default_rng(5)
    x = (rng.standard_normal((1, 1, n)) + 1j * rng.standard_normal((1, 1, n)))
    y = (rng.standard_normal((1, 1, n)) + 1j * rng.standard_normal((1, 1, n)))
    noise = (rng.standard_normal((1, 2, n)) + 1j * rng.standard_normal((1, 2, n)))
    f = _lib.DeviceField(ctx, n, 1, 1, precision=_lib.PMX_F32)
    f.upload(x, y)
    _lib.ampliflat_exec(ctx, f, 4.0, [0.25], noise=noise)
    gx, gy = f.download()
    np.testing.assert_allclose(gx[0, 0], 2.0 * x[0, 0] + 0.25 * noise[0, 0], rtol=0, atol=2e-6)
    np.testing.assert_allclose(gy[0, 0], 2.0 * y[0, 0] + 0.25 * noise[0, 1], rtol=0, atol=2e-6)


def test_fp32_qpsk_count_is_fp64_only():
    from polmux_b200 import _lib
    ctx = _lib.default_context()
    f = _lib.DeviceField(ctx, 1 << 12, 1, 1, precision=_lib.PMX_F32)
    with pytest.raises(_lib.PolmuxError):
        _lib.qpsk_count(ctx, f, np.zeros((2, 256), dtype=np.uint8), 256, 16, 0)
