"""PMD-aware digital backpropagation (pmx_dbp_desc.pmd, pmx_dbp_set_plates, dbp(brf=...), McRunner(compensation='dbp_pmd')).

The oracle is tests/dbp_oracle.dbp_pmd, built from the pinned forward oracle's checkstep, matrix_step and matrix_nl_step.
It is tied to the forward oracle by the exact-inverse property on 'gps-' links (with the forward run's own steps and
xi = 1, DBP returns the Tx field) and to the pinned inverse_pmd by the linear limit (xi = 0, one step per span)."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest

import oracle.fiber_oracle as orc
import dbp_oracle
import polmux_b200 as pmx
from polmux_b200 import _lib, mc
from polmux_b200.dbp import dbp_plan
from polmux_b200.fiber import fiber_setup, setup_to_desc
from common import _cols, _mc_scenario, base_fiber, make_tx, rel_l2

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GAIN_DB = 16.0


def _setup(nsymb, nt, nch=1, ftype='unique', pavg_mw=4.0, length=8e4, manakov=False, nplates=20, dgd=0.5, dphimax=0.02,
           **extra):
    """-> (oracle GState with the Tx field, product FiberSetup of the 'gps-' fiber with its plates in s.brf)"""
    gs = make_tx(nsymb, nt, nch=nch, ftype=ftype, pavg_mw=pavg_mw)
    fib = base_fiber(length=length, slope=0.057, dphimax=dphimax, dgd=dgd, nplates=nplates,
                     manakov='yes' if manakov else 'no', **extra)
    s = fiber_setup(fib, 'gps-', rng=np.random.Generator(np.random.PCG64(7)))
    return gs, s


def _brfs(s, nspan, batch=1):
    """nspan plate draws, [span][realization]: the setup's own plates first, fresh draws for the rest"""
    out = []
    for k in range(nspan):
        row = []
        for b in range(batch):
            if k == 0 and b == 0:
                row.append({x: np.asarray(s.brf[x], dtype=np.float64) for x in ('db0', 'theta', 'epsilon')})
            else:
                d = mc.draw_plates(mc.plate_seed(b, k), s.nplates)
                row.append(dict(zip(('db0', 'theta', 'epsilon'), d)))
        out.append(row)
    return out


def _plates(brfs):
    """[span][realization] brfs -> (db0, theta, epsilon), each [nspan][plate_sets][nplates]"""
    return tuple(np.array([[b[x] for b in row] for row in brfs]) for x in ('db0', 'theta', 'epsilon'))


def _forward(ux, uy, s, brfs, gain):
    """noise-free 'gps-' link of the oracle: span k through brfs[k] -> (ux, uy, steps of every span, schedules)"""
    steps, scheds = [], []
    for b in brfs:
        _, _, ux, uy, _, sched = orc.matrix_ssfm(ux, uy, s.betat, s.db1, s.dzmaxt, s.dphimaxt, s.gam, s.alphalin, s.nfc,
                                                 s.length, s.nplates, 'yes' if s.manakov else 'no', s.fls, b)
        steps.append([st['dz'] for st in sched])
        scheds.append(sched)
        if gain is not None:
            ux, uy = ux * math.sqrt(gain), uy * math.sqrt(gain)
    return ux, uy, steps, scheds


def _oracle(ux, uy, s, brfs, real=np.float64, **kw):
    return dbp_oracle.dbp_pmd(ux, uy, s.betat, s.db1, s.gam, s.alphalin, s.nfc, s.length, 'yes' if s.manakov else 'no',
                              brfs, real=real, **kw)


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize('case', ['straddle', 'one_step_100_plates', 'ten_plates_40_steps'])
def test_partition_replica_equals_the_forward_schedule(case):
    """the oracle's replica of the forward partition, fed with a forward run's own steps, is that run's sched exactly"""
    if case == 'straddle':
        gs, s = _setup(256, 16, pavg_mw=8.0, nplates=20)
    elif case == 'one_step_100_plates':
        gs, s = _setup(256, 16, nplates=100, dphimax=math.inf, dzmax=8e4)
    else:
        gs, s = _setup(256, 16, pavg_mw=30.0, nplates=10, length=1e5, dphimax=0.07)
    _, _, steps, scheds = _forward(gs.FIELDX, gs.FIELDY, s, [s.brf], None)
    n = len(steps[0])
    if case == 'straddle':
        assert n > 2 and any(st['nmem'] for st in scheds[0])
    elif case == 'one_step_100_plates':
        assert n == 1 and scheds[0][0]['ntrunk'] == 100
    else:
        assert 30 <= n <= 60, n
    rep = dbp_oracle.forward_partition(steps[0], s.length, s.nplates)
    assert [(r['ntrunk'], r['nmem'], r['ntot'], r['dzb']) for r in rep] == \
           [(r['ntrunk'], r['nmem'], r['ntot'], r['dzb']) for r in scheds[0]]


@pytest.mark.parametrize('manakov', [False, True])
@pytest.mark.parametrize('nch', [1, 3])
def test_oracle_dbp_pmd_inverts_the_forward_link(manakov, nch):
    """forward 'gps-' over two spans with a 16 dB gain and different plates per span, then PMD-aware DBP with the forward
    steps and xi = 1: the Tx field back"""
    gs, s = _setup(256, 16, nch=nch, ftype='sepfields' if nch > 1 else 'unique', manakov=manakov)
    g = 10 ** (GAIN_DB / 10)
    brfs = [r[0] for r in _brfs(s, 2)]
    ux, uy, steps, _ = _forward(gs.FIELDX, gs.FIELDY, s, brfs, g)
    assert sum(len(x) for x in steps) > 4
    bx, by = _oracle(ux, uy, s, brfs, nspan=2, gain=g, step_len=np.concatenate(steps), span_steps=[len(x) for x in steps])
    err = rel_l2(bx, by, gs.FIELDX, gs.FIELDY)
    assert err <= 1e-12, err


def test_oracle_linear_limit_is_inverse_pmd():
    """xi = 0 and one step per span: the pinned inverse_pmd of the spans' fibers, times (exp(alpha*L/2)/sqrt(G))^nspan"""
    gs, s = _setup(256, 16)
    g = 10 ** (GAIN_DB / 10)
    brfs = [r[0] for r in _brfs(s, 2)]
    bx, by = _oracle(gs.FIELDX, gs.FIELDY, s, brfs, nspan=2, gain=g, steps_per_span=1, xi=0.0)
    wx, wy = dbp_oracle.inverse_pmd_chain(gs.FIELDX, gs.FIELDY, brfs, s.betat, s.db1, s.length, s.alphalin, gain=g)
    err = rel_l2(bx, by, wx, wy)
    assert err <= 1e-12, err


def _create(desc, **kw):
    lib = _lib.load()
    nspan, gain = kw.pop('nspan', 1), kw.pop('gain', 0.0)
    d, dk = _lib.make_dbp(nspan, gain, **kw)
    rc = lib.pmx_dbp_create(None, ctypes.byref(desc), ctypes.byref(d), ctypes.byref(ctypes.c_void_p()))
    return rc, lib.pmx_last_error(None).decode()


def test_dbp_pmd_create_rejects_what_it_cannot_run():
    """pmx_dbp_create with pmd = 1 checks the fiber and the schedule before it needs a context"""
    make_tx(256, 16)
    s = fiber_setup(base_fiber(), 'g-s-')
    desc, keep = setup_to_desc(s)
    rc, msg = _create(desc, steps_per_span=2, pmd=True)
    assert rc == _lib.PMX_ERR_INVALID and "'p' flag" in msg, msg
    _, sp = _setup(256, 16, nplates=10)
    desc, keep = setup_to_desc(sp)
    desc.nplates = 0
    rc, msg = _create(desc, steps_per_span=2, pmd=True)
    assert rc == _lib.PMX_ERR_INVALID and 'nplates' in msg, msg
    desc.nplates = 10
    L = sp.length
    rc, msg = _create(desc, step_len=[L * (1 + 5e-10), 0.0], pmd=True)    # a step past the last plate (fiber.m:910)
    assert rc == _lib.PMX_ERR_PLATE_INDEX and 'plate' in msg, msg
    rc, msg = _create(desc, steps_per_span=200000, nspan=10, pmd=True)    # 2e6 steps of 2.8 KB packages
    assert rc == _lib.PMX_ERR_INVALID and '1 GiB' in msg, msg
    rc, msg = _create(desc, steps_per_span=4, nspan=2, pmd=True)          # valid: only the context is missing
    assert rc == _lib.PMX_ERR_INVALID and 'null context' in msg, msg
    with pytest.raises(ValueError):
        dbp_plan(None, s, plates=(np.zeros((1, 1, 1)),) * 3)


def test_mc_run_rejects_pmd_blind_dbp_without_a_receive_chain():
    """pmx_mc_desc.dbp with pmd = 0 and no receive chain: the data-aided decision needs the PMD undone"""
    lib = _lib.load()
    make_tx(256, 16)
    s = fiber_setup(base_fiber(), 'g-s-')
    desc, keep = setup_to_desc(s)
    d, dk = _lib.make_dbp(1, 0.0, steps_per_span=1)
    devs = (ctypes.c_int32 * 1)(0)
    sym = np.zeros((2, 256), np.uint8)
    m = _lib.McDesc()
    m.ndev, m.device_ids, m.nreal, m.batch, m.nspan = 1, devs, 1, 1, 1
    m.sym, m.nsymb, m.nt = sym.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), 256, 16
    m.dbp = ctypes.pointer(d)
    x = np.zeros((1, 1, 4096), np.complex128)
    io = _lib.complex_field(x, x.copy())
    err = ctypes.create_string_buffer(512)
    counts = np.zeros(1, np.int64)
    rc = lib.pmx_mc_run(ctypes.byref(desc), ctypes.byref(m), ctypes.byref(io), counts.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)),
                        None, err, 512)
    assert rc == _lib.PMX_ERR_INVALID and 'PMD-aware' in err.value.decode(), err.value


def test_dbp_pmd_structs_match_the_header(tmp_path):
    """gcc probe against the header: the appended fields of pmx_dbp_desc and pmx_mc_desc equal their ctypes mirrors"""
    structs = {'pmx_dbp_desc': _lib.DbpDesc, 'pmx_mc_desc': _lib.McDesc}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "polmux_ssfm.h"', 'int main(void){']
    for cname, cls in structs.items():
        lines.append('printf("%s %%zu\\n", sizeof(%s));' % (cname, cname))
        for fname, _ in cls._fields_:
            lines.append('printf("%s.%s %%zu\\n", offsetof(%s, %s));' % (cname, fname, cname, fname))
    lines.append('return 0;}')
    src = tmp_path / 'probe.c'
    src.write_text('\n'.join(lines))
    exe = tmp_path / 'probe'
    subprocess.run(['gcc', '-I', os.path.join(ROOT, 'include'), str(src), '-o', str(exe)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    for cname, cls in structs.items():
        assert int(out[cname]) == ctypes.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert int(out['%s.%s' % (cname, fname)]) == getattr(cls, fname).offset, (cname, fname)
    assert _lib.DbpDesc.reserved.offset == ctypes.sizeof(_lib.DbpDesc) - 4 and _lib.DbpDesc.pmd.offset == _lib.DbpDesc.gain.offset + 8
    assert _lib.McDesc.dbp.offset == ctypes.sizeof(_lib.McDesc) - ctypes.sizeof(ctypes.c_void_p)   # appended


def test_mc_runner_takes_dbp_pmd_with_the_genie_receiver():
    """'dbp_pmd' passes McRunner's checks with 'genie' (it fails later, on the missing context); 'dbp' still raises"""
    make_tx(256, 16)
    s = fiber_setup(base_fiber(), 'g-s-')
    args = (None, s, None, None, np.zeros((2, 256), np.uint8), 256, 16, 1, 16.0, 5.0, 2, 2)
    with pytest.raises(ValueError):
        mc.McRunner(*args, receiver='genie', compensation='dbp')
    with pytest.raises(Exception) as e:
        mc.McRunner(*args, receiver='genie', compensation='dbp_pmd')
    assert not isinstance(e.value, ValueError), e.value


# ---------------------------------------------------------------------------------------------------------------- GPU
def _run_device(ctx, s, xs, ys, plates, precision='f64', **kw):
    """PMD-aware DBP of the fields xs, ys ([batch][nfc][nfft]) on the device -> (x, y) of the same shape"""
    b = xs.shape[0]
    fld = _lib.DeviceField(ctx, s.nfft, s.nfc, b, precision={'f64': _lib.PMX_F64, 'f32': _lib.PMX_F32}[precision])
    fld.upload(xs, ys)
    plan = dbp_plan(ctx, s, batch=b, precision=precision, plates=plates, **kw)
    plan.execute(fld)
    plan.close()
    out = fld.download()
    fld.close()
    return out


PARITY = [  # nsymb, nt, nch, manakov, schedule, nspan, batch, nplates
    (256, 16, 1, False, 'uniform', 3, 1, 20),
    (256, 16, 3, True, 'explicit', 1, 1, 20),
    (4096, 16, 1, True, 'explicit', 3, 1, 20),
    (4096, 16, 1, False, 'one_step', 1, 1, 100),
    (65536, 16, 1, True, 'uniform', 1, 2, 20),
    (65536, 16, 1, False, 'one_step', 2, 2, 100),
]


@pytest.mark.gpu
@pytest.mark.parametrize('case', PARITY, ids=lambda c: '%dx%d-nfc%d-%s-%s-%dspan-b%d-%dpl' % (c[0], c[1], c[2], 'man' if c[3] else 'cnlse', c[4], c[5], c[6], c[7]))
def test_dbp_pmd_matches_the_oracle_fp64(ctx, case):
    nsymb, nt, nch, manakov, sched, nspan, batch, nplates = case
    gs, s = _setup(nsymb, nt, nch=nch, ftype='sepfields' if nch > 1 else 'unique', manakov=manakov, nplates=nplates)
    g = 10 ** (GAIN_DB / 10) if nspan > 1 else None
    if sched == 'uniform':
        kw = dict(steps_per_span=5)
    elif sched == 'one_step':
        kw = dict(steps_per_span=1)
    else:
        rng = np.random.default_rng(nsymb + nspan)
        steps = [list(np.diff(np.concatenate([[0.0], np.sort(rng.random(3 + k)) * s.length, [s.length]]))) for k in range(nspan)]
        kw = dict(step_len=np.concatenate(steps), span_steps=[len(x) for x in steps])
    brfs = _brfs(s, nspan, batch)                                            # per-realization plates when batch > 1
    xs = np.concatenate([_cols(gs.FIELDX), _cols(np.roll(gs.FIELDX, 7, axis=0) * 1j)][:batch])
    ys = np.concatenate([_cols(gs.FIELDY), _cols(np.roll(gs.FIELDY, -5, axis=0))][:batch])
    gx, gy = _run_device(ctx, s, xs, ys, _plates(brfs), nspan=nspan, gain_db=GAIN_DB if g else None, **kw)
    errs = []
    for b in range(batch):
        wx, wy = _oracle(xs[b].T, ys[b].T, s, [row[b] for row in brfs], nspan=nspan, gain=g, **kw)
        errs.append(rel_l2(gx[b].T, gy[b].T, wx, wy))
    print('dbp pmd parity %s: rel_l2 %s' % (case, ['%.3e' % e for e in errs]))
    assert max(errs) <= 1e-10, errs


@pytest.mark.gpu
def test_dbp_pmd_matches_the_oracle_fp32(ctx):
    gs, s = _setup(256, 16, manakov=True)
    brfs = _brfs(s, 2)
    g = 10 ** (GAIN_DB / 10)
    gx, gy = _run_device(ctx, s, _cols(gs.FIELDX), _cols(gs.FIELDY), _plates(brfs), precision='f32', nspan=2,
                         gain_db=GAIN_DB, steps_per_span=10)
    wx, wy = _oracle(gs.FIELDX, gs.FIELDY, s, [r[0] for r in brfs], nspan=2, gain=g, steps_per_span=10)
    err = rel_l2(gx[0].T, gy[0].T, wx, wy)
    print('dbp pmd parity fp32: rel_l2 %.3e' % err)
    assert err <= 1e-5


@pytest.mark.gpu
def test_dbp_pmd_vector_dispersion_mode_matches_the_oracle(ctx):
    """betat and db1 uploaded per bin (disp_mode='vector'): pass B of every step reads the plan's negated db1 table"""
    gs, s = _setup(256, 16, manakov=True)
    brfs = _brfs(s, 2)
    g = 10 ** (GAIN_DB / 10)
    gx, gy = _run_device(ctx, s, _cols(gs.FIELDX), _cols(gs.FIELDY), _plates(brfs), nspan=2, gain_db=GAIN_DB,
                         steps_per_span=5, disp_mode='vector')
    wx, wy = _oracle(gs.FIELDX, gs.FIELDY, s, [r[0] for r in brfs], nspan=2, gain=g, steps_per_span=5)
    err = rel_l2(gx[0].T, gy[0].T, wx, wy)
    print('dbp pmd parity, vector dispersion mode: rel_l2 %.3e' % err)
    assert err <= 1e-10


@pytest.mark.gpu
@pytest.mark.parametrize('case', ['c1', 'c2_span'])
def test_dbp_pmd_inverts_fiber_on_the_device(case):
    """pmx.fiber(fib, 'gps-', trace=True) then pmx.dbp(fib, 'gps-', step_len=trace_dz, brf=brf): the Tx field back.
    C1: 2^16, CNLSE, 10 plates, 100 km; a C2 span: 2^20, Manakov, 100 plates, 80 km"""
    if case == 'c1':
        make_tx(4096, 16)
        fib = base_fiber(length=1e5, dgd=1.0, nplates=10, manakov='no')
    else:
        make_tx(65536, 16)
        fib = base_fiber(length=8e4, dgd=0.3, nplates=100, manakov='yes')
    G = pmx.GSTATE
    tx, ty = G.FIELDX_TX.copy(), G.FIELDY_TX.copy()
    brf = pmx.fiber(fib, 'gps-', trace=True, rng=np.random.Generator(np.random.PCG64(11)))
    dz, ntr = np.asarray(pmx.FIBER_LAST['trace_dz']), np.asarray(pmx.FIBER_LAST['trace_ntrunk'])
    assert len(dz) > 1
    rep = dbp_oracle.forward_partition(dz, float(fib['length']), int(fib['nplates']))
    assert [r['ntrunk'] for r in rep] == list(ntr)
    pmx.dbp(fib, 'gps-', step_len=dz, brf=brf)
    err = rel_l2(G.FIELDX, G.FIELDY, tx, ty)
    print('dbp pmd exact inverse %s: %d steps, rel_l2 %.3e' % (case, len(dz), err))
    assert err <= 1e-11


@pytest.mark.gpu
def test_dbp_pmd_inverts_a_two_span_link_on_the_device(ctx):
    """two 'gps-' spans with a new plate draw each and a noise-free 16 dB amplifier after each, through the resident
    plan API; DBP with both spans' trace_dz and plates returns the Tx field"""
    make_tx(4096, 16)
    G = pmx.GSTATE
    s = fiber_setup(base_fiber(length=8e4, dgd=0.5, nplates=20, manakov='yes'), 'gps-',
                    rng=np.random.Generator(np.random.PCG64(3)))
    brfs = _brfs(s, 2)
    gain = 10 ** (GAIN_DB / 10)
    desc, keep = setup_to_desc(s)
    fld = _lib.DeviceField(ctx, s.nfft, 1, 1)
    fld.upload(G.FIELDX_TX, G.FIELDY_TX)
    plan = _lib.Plan(ctx, desc, keep)
    steps = []
    for k in range(2):
        b = brfs[k][0]
        plan.set_plates(b['db0'], b['theta'], b['epsilon'])
        dz, ntr = plan.execute(fld, trace_cap=1 << 14).schedule(0)
        assert [r['ntrunk'] for r in dbp_oracle.forward_partition(dz, s.length, s.nplates)] == list(ntr)
        steps.append(dz)
        _lib.ampliflat_exec(ctx, fld, gain, [0.0])
    plan.close()
    dbp_plan(ctx, s, nspan=2, gain_db=GAIN_DB, step_len=np.concatenate(steps), span_steps=[len(x) for x in steps],
             plates=_plates(brfs)).execute(fld)
    x, y = fld.download()
    fld.close()
    err = rel_l2(x[0, 0], y[0, 0], G.FIELDX_TX[:, 0], G.FIELDY_TX[:, 0])
    print('dbp pmd exact inverse, two spans: %s steps, rel_l2 %.3e' % ([len(x) for x in steps], err))
    assert err <= 1e-11


@pytest.mark.gpu
def test_dbp_pmd_realizations_are_independent(ctx):
    """PMD-aware DBP of a batch (per-realization plates) equals, bit for bit, DBP of each realization alone (2^20: the
    batch runs as two stream groups)"""
    gs, s = _setup(65536, 16, manakov=True)
    brfs = _brfs(s, 2, 3)
    xs = np.concatenate([_cols(np.roll(gs.FIELDX, 11 * b, axis=0)) for b in range(3)])
    ys = np.concatenate([_cols(np.roll(gs.FIELDY, -3 * b, axis=0)) for b in range(3)])
    kw = dict(nspan=2, gain_db=GAIN_DB, steps_per_span=3)
    bx, by = _run_device(ctx, s, xs, ys, _plates(brfs), **kw)
    for b in range(3):
        ox, oy = _run_device(ctx, s, xs[b:b + 1], ys[b:b + 1], _plates([[row[b]] for row in brfs]), **kw)
        assert np.array_equal(ox[0], bx[b]) and np.array_equal(oy[0], by[b]), b


@pytest.mark.gpu
def test_dbp_pmd_linear_limit_is_the_genie_equaliser(ctx):
    """xi = 0 and one step per span: Link.equalize on the same field, times (exp(alpha*L/2)/sqrt(G))^nspan"""
    gs, s = _setup(4096, 16, manakov=True, nplates=20)
    nspan, batch = 2, 2
    link = mc.Link(ctx, s, nspan, batch, GAIN_DB, None)
    xs = np.concatenate([_cols(gs.FIELDX), _cols(np.roll(gs.FIELDX, 5, axis=0))])
    ys = np.concatenate([_cols(gs.FIELDY), _cols(np.roll(gs.FIELDY, 9, axis=0))])
    fld = _lib.DeviceField(ctx, s.nfft, 1, batch)
    fld.upload(xs, ys)
    link.equalize(fld)
    ex, ey = fld.download()
    fld.close()
    plates = tuple(np.stack([pl[i] for pl in link.plates]) for i in range(3))
    gx, gy = _run_device(ctx, s, xs, ys, plates, nspan=nspan, gain_db=GAIN_DB, steps_per_span=1, xi=0.0)
    sc = (math.exp(0.5 * s.alphalin * s.length) / math.sqrt(10 ** (GAIN_DB / 10))) ** nspan
    for b in range(batch):
        err = rel_l2(gx[b, 0], gy[b, 0], ex[b, 0] * sc, ey[b, 0] * sc)
        print('dbp pmd linear limit vs Link.equalize, realization %d: rel_l2 %.3e' % (b, err))
        assert err <= 1e-12


@pytest.mark.gpu
@pytest.mark.parametrize('receiver', ['genie', 'cohmix'])
def test_mc_with_dbp_pmd_python_and_native_agree(ctx, receiver):
    """McRunner(compensation='dbp_pmd') and run_mc_native(..., dbp_params={'pmd': True, ...}) count the same errors,
    realization by realization, on a small seeded job (16 realizations, 2 spans at 2^16, 20 plates)"""
    nsymb, nt, nspan, nreal, batch = 1 << 12, 16, 2, 16, 4
    G, setup, sym = _mc_scenario(nsymb, nt, 8.0)
    x = {'oftype': 'gauss', 'obw': 1.9, 'eftype': 'bessel5', 'ebw': 0.65, 'lopower': 0.0}
    dspp = dict(mu=1 / 2000, freqavg=200) if receiver == 'cohmix' else None
    dbpp = dict(steps_per_span=4)
    r = mc.McRunner(ctx, setup, G.FIELDX_TX, G.FIELDY_TX, sym, nsymb, nt, nspan, 16.0, 5.0, nreal, batch, receiver=receiver,
                    dsp_params=dspp, rx_params=x if receiver == 'cohmix' else None, compensation='dbp_pmd', dbp_params=dbpp)
    want, _ = r.run(ase_seed=3)
    r.close()
    got, _ = mc.run_mc_native(setup, G.FIELDX_TX, G.FIELDY_TX, sym, nsymb, nt, nspan, 16.0, 5.0, nreal, batch, devices=(0,),
                              ase_seed=3, receiver=x if receiver == 'cohmix' else None, dsp_params=dspp,
                              dbp_params=dict(dbpp, pmd=True))
    print('mc dbp_pmd %s counts %s' % (receiver, want.tolist()))
    assert np.array_equal(got, want), (got, want)


@pytest.mark.gpu
def test_dbp_pmd_plan_checks_its_plates(ctx):
    """pmx_dbp_exec before pmx_dbp_set_plates, and plate_sets other than 1 or batch: PMX_ERR_INVALID with a message"""
    gs, s = _setup(256, 16, nplates=10)
    desc, keep = setup_to_desc(s, batch=2)
    d, dk = _lib.make_dbp(1, 0.0, steps_per_span=2, pmd=True)
    plan = _lib.DbpPlan(ctx, desc, keep, d, dk)
    fld = _lib.DeviceField(ctx, s.nfft, 1, 2)
    with pytest.raises(_lib.PolmuxError) as e:
        plan.execute(fld)
    assert e.value.code == _lib.PMX_ERR_INVALID and 'pmx_dbp_set_plates' in str(e.value)
    z = np.zeros((1, 3, 10))
    with pytest.raises(_lib.PolmuxError) as e:
        plan.set_plates(z, z, z, plate_sets=3)
    assert e.value.code == _lib.PMX_ERR_INVALID and 'plate_sets' in str(e.value)
    plan.close()
    fld.close()
