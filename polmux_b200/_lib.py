"""ctypes binding of the C ABI in include/polmux_ssfm.h.

The shared library is built in-tree by ``__graft_entry__.build()`` (or ``make -C
polmux_b200/csrc``).  There is no fallback: if the library is missing or no
B200 is visible, every compute entry point raises ``PolmuxError``.
"""
from __future__ import annotations

import ctypes as C
import sys
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# POLMUX_SSFM_LIB: another build of the same CUDA library (e.g. the index-assert build of `make -C polmux_b200/csrc debug`)
LIB_PATH = os.environ.get('POLMUX_SSFM_LIB') or os.path.join(_HERE, 'lib', 'libpolmux_ssfm.so')

PMX_OK = 0
PMX_ERR_INVALID, PMX_ERR_UNSUPPORTED, PMX_ERR_CUDA = -1, -2, -3
PMX_ERR_PLATE_INDEX, PMX_ERR_NUMERIC, PMX_ERR_XPM_VECTOR = -4, -5, -6
PMX_F64, PMX_F32 = 0, 1
PMX_PLANAR, PMX_COMPLEX = 0, 1

# every symbol include/polmux_ssfm.h declares (checked by tests/test_abi.py)
EXPORTS = [
    'pmx_version', 'pmx_device_count', 'pmx_ctx_create', 'pmx_ctx_destroy', 'pmx_last_error',
    'pmx_ctx_sync', 'pmx_ctx_stream', 'pmx_fiber_run', 'pmx_field_create', 'pmx_field_destroy',
    'pmx_field_upload', 'pmx_field_download', 'pmx_field_broadcast', 'pmx_field_device_ptr',
    'pmx_plan_create', 'pmx_plan_destroy', 'pmx_plan_set_plates', 'pmx_fiber_exec',
    'pmx_ctx_launch_count', 'pmx_ampliflat_exec', 'pmx_count_errors', 'pmx_ctx_profile',
    'pmx_ctx_profile_read', 'pmx_qpsk_count', 'pmx_scalar_nl_exec', 'pmx_plan_set_length', 'pmx_field_max_power',
    'pmx_field_maxdiff2', 'pmx_field_lincomb', 'pmx_link_exec', 'pmx_link_run', 'pmx_field_mux', 'pmx_ampliflat_exec_pol',
    'pmx_host_is_pinned', 'pmx_scalar_adaptive_run', 'pmx_mc_run', 'pmx_mc_nccl_available',
    'pmx_ampliflat_exec_at', 'pmx_dsp_count', 'pmx_field_mean_power', 'pmx_pmd_matrix', 'pmx_field_jones', 'pmx_filter_create', 'pmx_field_copy_cols', 'pmx_field_modulate',
    'pmx_cohmix_exec', 'pmx_field_mean_power_xy', 'pmx_cohmix_run', 'pmx_dsp_phases', 'pmx_field_quantize', 'pmx_inverse_pmd_run',
    'pmx_dbp_create', 'pmx_dbp_exec', 'pmx_dbp_set_plates', 'pmx_dbp_channel_create', 'pmx_dbp_set_filter',
    'pmx_dbp_set_taps',
]


class PolmuxError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__('polmux_ssfm error %d: %s' % (code, msg))
        self.code = code


_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)


class FiberDesc(C.Structure):
    _fields_ = [
        ('nfft', C.c_int64), ('nfc', C.c_int32), ('batch', C.c_int32), ('precision', C.c_int32),
        ('manakov', C.c_int32), ('length', C.c_double), ('alphalin', C.c_double),
        ('dzmaxt', C.c_double), ('dphimaxt', C.c_double), ('gam', _dp), ('fls', C.c_int32 * 4),
        ('nplates', C.c_int32), ('plate_sets', C.c_int32), ('db0', _dp), ('theta', _dp),
        ('epsilon', _dp), ('betat', _dp), ('db1', _dp),
        ('disp_mode', C.c_int32), ('nsymb', C.c_int32), ('nt', C.c_int32), ('scalar_field', C.c_int32),
        ('symbolrate', C.c_double), ('b30', C.c_double), ('dgdrms', C.c_double), ('beta1', _dp), ('beta2', _dp),
        ('z_start', C.c_double), ('dz_first', C.c_double),
    ]


class Field(C.Structure):
    _fields_ = [('layout', C.c_int32), ('reserved', C.c_int32), ('xr', _dp), ('xi', _dp),
                ('yr', _dp), ('yi', _dp)]


class FiberResult(C.Structure):
    _fields_ = [('firstdz', _dp), ('ncycle', _ip), ('ntot', _ip), ('status', _ip),
                ('trace_dz', _dp), ('trace_ntrunk', _ip), ('trace_cap', C.c_int32)]


class DspDesc(C.Structure):
    _fields_ = [('nsymb', C.c_int32), ('nt', C.c_int32), ('apply_cma', C.c_int32), ('taps', C.c_int32), ('mu', C.c_double),
                ('R', C.c_double * 2), ('phizero', C.c_double), ('max_passes', C.c_int32), ('modorder', C.c_int32),
                ('freqavg', C.c_int32), ('phasavg', C.c_int32), ('poworder', C.c_int32), ('sample_shift', C.c_int32),
                ('peak', C.c_double), ('apply_easi', C.c_int32), ('easi_max_passes', C.c_int32), ('easi_mu', C.c_double),
                ('easi_phizero', C.c_double), ('easi_passes', C.POINTER(C.c_int32)), ('nlr_alpha', C.c_double), ('dcf_h', _dp), ('decim_ntaps', C.c_int32), ('reserved2', C.c_int32), ('decim_taps', _dp)]


class DbpDesc(C.Structure):
    _fields_ = [('nspan', C.c_int32), ('steps_per_span', C.c_int32), ('span_steps', _ip), ('step_len', _dp),
                ('xi', C.c_double), ('gain', C.c_double), ('pmd', C.c_int32), ('reserved', C.c_int32)]


class DbpBand(C.Structure):
    _fields_ = [('shift', C.c_int64), ('decim', C.c_int32), ('reserved', C.c_int32)]


class McReceiver(C.Structure):
    _fields_ = [('hf_opt', _dp), ('hf_el', _dp), ('lo_ecw', C.c_double), ('lo_detune', C.c_double), ('lo_phase', _dp),
                ('balanced', C.c_int32), ('reserved', C.c_int32), ('dsp', DspDesc), ('ref_patmat', C.POINTER(C.c_uint8)),
                ('dbp', C.POINTER(DbpDesc))]


class McDesc(C.Structure):
    _fields_ = [('ndev', C.c_int32), ('device_ids', C.POINTER(C.c_int32)), ('nreal', C.c_int32), ('batch', C.c_int32),
                ('nspan', C.c_int32), ('equalize', C.c_int32), ('db0', _dp), ('theta', _dp), ('epsilon', _dp),
                ('gain', C.c_double), ('sigma', _dp), ('ase_seed', C.c_uint64), ('sym', C.POINTER(C.c_uint8)),
                ('nsymb', C.c_int32), ('nt', C.c_int32), ('rx', C.POINTER(McReceiver)), ('dbp', C.POINTER(DbpDesc))]


class BrfDesc(C.Structure):
    _fields_ = [('ntrunk', C.c_int32), ('reserved', C.c_int32), ('lcorr', C.c_double), ('db0', _dp), ('theta', _dp),
                ('epsilon', _dp), ('betat', _dp), ('db1', _dp)]


class LinkDesc(C.Structure):
    _fields_ = [('nspan', C.c_int32), ('plate_sets', C.c_int32), ('db0', _dp), ('theta', _dp), ('epsilon', _dp),
                ('gain', C.c_double), ('sigma', _dp), ('noise', _dp), ('seeds', C.POINTER(C.c_uint64)),
                ('realization0', C.c_uint64), ('asepol', C.c_int32), ('reserved', C.c_int32)]


_lib = None


def load():
    """Load the shared library (once).  Raises PolmuxError if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PolmuxError(PMX_ERR_CUDA, 'CUDA library %s is not built; run __graft_entry__.build() '
                          '(there is no CPU fallback)' % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    lib.pmx_version.restype = C.c_int
    lib.pmx_device_count.restype = C.c_int
    lib.pmx_ctx_create.argtypes = [C.POINTER(vp), C.c_int]
    lib.pmx_ctx_destroy.argtypes = [vp]
    lib.pmx_ctx_destroy.restype = None
    lib.pmx_last_error.argtypes = [vp]
    lib.pmx_last_error.restype = C.c_char_p
    lib.pmx_ctx_sync.argtypes = [vp]
    lib.pmx_ctx_stream.argtypes = [vp]
    lib.pmx_ctx_stream.restype = vp
    lib.pmx_ctx_launch_count.argtypes = [vp]
    lib.pmx_ctx_launch_count.restype = C.c_int64
    lib.pmx_ctx_profile.argtypes = [vp, C.c_int]
    lib.pmx_ctx_profile_read.argtypes = [vp, _dp, C.POINTER(C.c_int64)]
    lib.pmx_fiber_run.argtypes = [vp, C.POINTER(FiberDesc), C.POINTER(Field), C.POINTER(FiberResult)]
    lib.pmx_field_create.argtypes = [vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.POINTER(vp)]
    lib.pmx_field_destroy.argtypes = [vp]
    lib.pmx_field_destroy.restype = None
    lib.pmx_field_upload.argtypes = [vp, C.POINTER(Field), C.c_int32, C.c_int32]
    lib.pmx_field_download.argtypes = [vp, C.POINTER(Field), C.c_int32, C.c_int32]
    lib.pmx_field_broadcast.argtypes = [vp, vp]
    lib.pmx_field_device_ptr.argtypes = [vp]
    lib.pmx_field_device_ptr.restype = vp
    lib.pmx_plan_create.argtypes = [vp, C.POINTER(FiberDesc), C.POINTER(vp)]
    lib.pmx_plan_destroy.argtypes = [vp]
    lib.pmx_plan_destroy.restype = None
    lib.pmx_plan_set_plates.argtypes = [vp, C.c_int32, _dp, _dp, _dp]
    lib.pmx_fiber_exec.argtypes = [vp, vp, C.POINTER(FiberResult)]
    lib.pmx_host_is_pinned.argtypes = [vp]
    lib.pmx_dsp_phases.argtypes = [vp, vp, C.POINTER(DspDesc), _dp, _dp, C.POINTER(C.c_int32)]
    lib.pmx_dsp_count.argtypes = [vp, vp, C.POINTER(DspDesc), C.POINTER(C.c_uint8), vp, C.POINTER(C.c_int32)]
    lib.pmx_mc_run.argtypes = [C.POINTER(FiberDesc), C.POINTER(McDesc), C.POINTER(Field), C.POINTER(C.c_int64),
                               C.POINTER(C.c_int64), C.c_char_p, C.c_int32]
    lib.pmx_scalar_adaptive_run.argtypes = [vp, C.POINTER(FiberDesc), C.c_double, C.c_double, C.c_int32, C.POINTER(Field),
                                            C.POINTER(FiberResult)]
    lib.pmx_ampliflat_exec.argtypes = [vp, vp, C.c_double, _dp, _dp, C.c_uint64]
    lib.pmx_ampliflat_exec_pol.argtypes = [vp, vp, C.c_double, _dp, _dp, C.c_uint64, C.c_int32]
    lib.pmx_count_errors.argtypes = [vp, vp, vp, C.c_int64, C.c_int32, vp]
    lib.pmx_qpsk_count.argtypes = [vp, vp, vp, C.c_int32, C.c_int32, vp]
    lib.pmx_scalar_nl_exec.argtypes = [vp, vp, _dp, C.c_double, C.c_double, C.c_int32, C.c_int32]
    lib.pmx_plan_set_length.argtypes = [vp, C.c_double]
    lib.pmx_field_max_power.argtypes = [vp, vp, _dp]
    lib.pmx_field_mean_power.argtypes = [vp, vp, _dp]
    lib.pmx_field_mean_power_xy.argtypes = [vp, vp, _dp, _dp]
    lib.pmx_pmd_matrix.argtypes = [vp, C.c_int64, C.c_int32, C.POINTER(BrfDesc), _dp, C.c_int32, _dp, _dp]
    lib.pmx_field_jones.argtypes = [vp, vp, _dp]
    lib.pmx_field_copy_cols.argtypes = [vp, C.c_int32, vp, C.c_int32, C.c_int32]
    lib.pmx_field_modulate.argtypes = [vp, vp, C.c_int64]
    lib.pmx_field_quantize.argtypes = [vp, vp, C.c_int32]
    lib.pmx_cohmix_exec.argtypes = [vp, vp, C.c_double, C.c_double, _dp, C.c_int32]
    lib.pmx_filter_create.argtypes = [vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _dp, C.c_int32, C.POINTER(vp)]
    lib.pmx_field_maxdiff2.argtypes = [vp, vp, vp, _dp]
    lib.pmx_field_lincomb.argtypes = [vp, vp, C.c_double, vp, C.c_double, vp]
    lib.pmx_field_mux.argtypes = [vp, C.POINTER(Field), C.c_int32, C.POINTER(C.c_int64), _dp, C.POINTER(C.c_int64),
                                  C.POINTER(C.c_int64)]
    lib.pmx_link_exec.argtypes = [vp, vp, C.POINTER(LinkDesc), C.POINTER(FiberResult)]
    lib.pmx_link_run.argtypes = [vp, C.POINTER(FiberDesc), C.POINTER(LinkDesc), C.POINTER(Field), C.POINTER(FiberResult)]
    lib.pmx_dbp_create.argtypes = [vp, C.POINTER(FiberDesc), C.POINTER(DbpDesc), C.POINTER(vp)]
    lib.pmx_dbp_exec.argtypes = [vp, vp]
    lib.pmx_dbp_set_plates.argtypes = [vp, C.c_int32, _dp, _dp, _dp]
    lib.pmx_dbp_set_filter.argtypes = [vp, C.c_double]
    lib.pmx_dbp_set_taps.argtypes = [vp, C.c_int32, _dp]
    lib.pmx_dbp_channel_create.argtypes = [vp, C.POINTER(FiberDesc), C.POINTER(DbpDesc), C.POINTER(DbpBand), C.POINTER(vp)]
    _lib = lib
    return lib


def pmd_matrix(ctx, nfft, brfs, mat=None, gvd=True, want_u=True, want_uinv=True):
    """-> (Uinv, U), each [2, 2, nfft] complex128 or None (pmx_pmd_matrix; inverse_pmd.m:73-131)"""
    keep, descs = [], (BrfDesc * len(brfs))()
    for d, b in zip(descs, brfs):
        arrs = {k: np.ascontiguousarray(np.asarray(b[k], dtype=np.float64).ravel()) for k in ('db0', 'theta', 'epsilon', 'betat', 'db1')}
        if arrs['betat'].size != nfft or arrs['db1'].size != nfft:
            raise ValueError('brf.betat / brf.db1 must have one value per frequency')
        if not (arrs['db0'].size == arrs['theta'].size == arrs['epsilon'].size):
            raise ValueError('brf.db0 / theta / epsilon must have one value per trunk')
        keep.append(arrs)
        d.ntrunk, d.lcorr = arrs['theta'].size, float(np.asarray(b['lcorr']).ravel()[0])
        for k, a in arrs.items():
            setattr(d, k, a.ctypes.data_as(_dp))
    m = None
    if mat is not None:
        mm = np.asarray(mat, dtype=np.complex128)
        if mm.shape != (2, 2):
            raise ValueError('options.mat must be a [2,2] matrix')
        m = np.ascontiguousarray(mm.reshape(4)).view(np.float64)
    u = np.zeros((nfft, 2, 2), dtype=np.complex128) if want_u else None          # memory order of U(2,2,Nfft)
    ui = np.zeros((nfft, 2, 2), dtype=np.complex128) if want_uinv else None
    ctx.check(ctx.lib.pmx_pmd_matrix(ctx.h, nfft, len(brfs), descs, None if m is None else m.ctypes.data_as(_dp),
                                     1 if gvd else 0, None if u is None else u.ctypes.data_as(_dp),
                                     None if ui is None else ui.ctypes.data_as(_dp)))
    tr = lambda a: None if a is None else a.transpose(2, 1, 0)                   # [n][j][i] -> (i, j, n)
    return tr(ui), tr(u)


def field_copy_cols(dst, dst_bc, src, src_bc, count=1):
    """count realization-columns of src (from src_bc) -> dst (from dst_bc), device to device"""
    dst.ctx.check(dst.ctx.lib.pmx_field_copy_cols(dst.h, int(dst_bc), src.h, int(src_bc), int(count)))


def field_quantize(ctx, field, bits):
    """ADC with `bits` bits on the currents in `field` (pmx_field_quantize, dsp4cohdec.m:157-162)"""
    ctx.check(ctx.lib.pmx_field_quantize(ctx.h, field.h, int(bits)))


def field_modulate(ctx, field, m):
    """u(n) <- u(n) * exp(+i*2*pi*m*n/nfft) (pmx_field_modulate)"""
    ctx.check(ctx.lib.pmx_field_modulate(ctx.h, field.h, int(m)))


def cohmix_exec(ctx, field, lo_ecw=1.0, lo_detune=0.0, lo_phase=None, balanced=True):
    """LO mixing + photodetection in place (pmx_cohmix_exec): each polarization becomes I_a + i*I_b"""
    ph = None if lo_phase is None else np.ascontiguousarray(np.asarray(lo_phase, dtype=np.float64).ravel())
    if ph is not None and ph.size != field.nfft:
        raise ValueError('Incompatible vector.')                               # receiver_cohmix.m:203-205
    ctx.check(ctx.lib.pmx_cohmix_exec(ctx.h, field.h, float(lo_ecw), float(lo_detune),
                                      None if ph is None else ph.ctypes.data_as(_dp), 1 if balanced else 0))


def field_jones(ctx, field, jones):
    """[ux; uy] <- J [ux; uy] on the device field (pmx_field_jones)"""
    j = np.ascontiguousarray(np.asarray(jones, dtype=np.complex128).reshape(4)).view(np.float64)
    ctx.check(ctx.lib.pmx_field_jones(ctx.h, field.h, j.ctypes.data_as(_dp)))


def field_mean_power(ctx, field):
    """-> [batch, nfc] mean |ux|^2 + |uy|^2 (pmx_field_mean_power)"""
    out = np.zeros((field.batch, field.nfc), dtype=np.float64)
    ctx.check(ctx.lib.pmx_field_mean_power(ctx.h, field.h, out.ctypes.data_as(_dp)))
    return out


def field_mean_power_xy(ctx, field):
    """-> (mean |ux|^2, mean |uy|^2), each [batch, nfc] (pmx_field_mean_power_xy)"""
    px = np.zeros((field.batch, field.nfc), dtype=np.float64)
    py = np.zeros_like(px)
    ctx.check(ctx.lib.pmx_field_mean_power_xy(ctx.h, field.h, px.ctypes.data_as(_dp), py.ctypes.data_as(_dp)))
    return px, py


def host_is_pinned(a) -> bool:
    """True when the numpy array lives in page-locked host memory (pmx_host_is_pinned)."""
    try:
        return bool(load().pmx_host_is_pinned(C.c_void_p(a.ctypes.data)))
    except Exception:
        return False


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _ptr(a):
    return a.ctypes.data_as(_dp) if a is not None else None


class Context:
    """One pmx_ctx (one GPU, one stream)."""

    def __init__(self, device: int = 0):
        self.lib = load()
        h = C.c_void_p()
        rc = self.lib.pmx_ctx_create(C.byref(h), int(device))
        if rc != PMX_OK:
            raise PolmuxError(rc, self.lib.pmx_last_error(None).decode())
        self.h = h
        self.device = device

    def check(self, rc):
        if rc != PMX_OK:
            raise PolmuxError(rc, self.lib.pmx_last_error(self.h).decode())

    def sync(self):
        self.check(self.lib.pmx_ctx_sync(self.h))

    @property
    def stream(self):
        return self.lib.pmx_ctx_stream(self.h)

    @property
    def launches(self):
        return int(self.lib.pmx_ctx_launch_count(self.h))

    def profile(self, enable: bool):
        self.check(self.lib.pmx_ctx_profile(self.h, 1 if enable else 0))

    def profile_read(self):
        ms = np.zeros(4)
        n = np.zeros(4, dtype=np.int64)
        self.check(self.lib.pmx_ctx_profile_read(self.h, _ptr(ms), n.ctypes.data_as(C.POINTER(C.c_int64))))
        return ms, n

    def close(self):
        if getattr(self, 'h', None):
            self.lib.pmx_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        # at interpreter shutdown objects die in no particular order (a context before its plans): leave them to the process exit
        if sys.is_finalizing():
            return
        try:
            self.close()
        except Exception:
            pass


_default_ctx = {}


def default_context(device: int = 0) -> Context:
    if device not in _default_ctx:
        _default_ctx[device] = Context(device)
    return _default_ctx[device]


def make_desc(nfft, nfc, batch, length, alphalin, dzmaxt, dphimaxt, gam, fls, manakov, nplates,
              db0, theta, epsilon, betat, db1, plate_sets=1, precision=PMX_F64, scalar=None, scalar_field=False,
              z_start=0.0, dz_first=0.0):
    """Build a FiberDesc plus the list of arrays that must stay alive while it is used.

    scalar: None (vector dispersion mode: betat/db1 cross the boundary) or a dict with nsymb, nt,
    symbolrate, b30, dgdrms, beta1, beta2 (scalar dispersion mode: betat/db1 stay on the host)."""
    keep = {}
    keep['gam'] = _f64(np.atleast_1d(gam))
    keep['db0'] = _f64(db0).reshape(-1)
    keep['theta'] = _f64(theta).reshape(-1)
    keep['epsilon'] = _f64(epsilon).reshape(-1)
    # betat / db1 arrive as [nfft, nfc] (column-major columns) -> [nfc][nfft]
    keep['betat'] = _f64(np.asarray(betat).reshape(nfft, nfc).T) if (betat is not None and scalar is None) else None
    keep['db1'] = _f64(np.asarray(db1).reshape(nfft, nfc).T) if (db1 is not None and scalar is None) else None
    d = FiberDesc()
    d.nfft, d.nfc, d.batch, d.precision = int(nfft), int(nfc), int(batch), int(precision)
    d.manakov = 1 if manakov else 0
    d.scalar_field = 1 if scalar_field else 0   # scalar_ssfm dispatch (fiber.m:372-380)
    d.z_start, d.dz_first = float(z_start), float(dz_first)   # resumed loop (x.dphiadapt, fiber.m:603-609)
    d.length, d.alphalin, d.dzmaxt, d.dphimaxt = float(length), float(alphalin), float(dzmaxt), float(dphimaxt)
    d.gam = _ptr(keep['gam'])
    d.fls = (C.c_int32 * 4)(*[int(v) for v in fls])
    d.nplates, d.plate_sets = int(nplates), int(plate_sets)
    d.db0, d.theta, d.epsilon = _ptr(keep['db0']), _ptr(keep['theta']), _ptr(keep['epsilon'])
    d.betat, d.db1 = _ptr(keep['betat']), _ptr(keep['db1'])
    if scalar is not None:
        keep['beta1'] = _f64(np.atleast_1d(scalar['beta1']))
        keep['beta2'] = _f64(np.atleast_1d(scalar['beta2']))
        d.disp_mode = 1
        d.nsymb, d.nt = int(scalar['nsymb']), int(scalar['nt'])
        d.symbolrate, d.b30, d.dgdrms = float(scalar['symbolrate']), float(scalar['b30']), float(scalar['dgdrms'])
        d.beta1, d.beta2 = _ptr(keep['beta1']), _ptr(keep['beta2'])
    return d, keep


class Result:
    def __init__(self, batch, trace_cap=0):
        self.firstdz = np.zeros(batch)
        self.ncycle = np.zeros(batch, dtype=np.int32)
        self.ntot = np.zeros(batch, dtype=np.int32)
        self.status = np.zeros(batch, dtype=np.int32)
        self.trace_cap = trace_cap
        self.trace_dz = np.zeros((batch, trace_cap)) if trace_cap else None
        self.trace_ntrunk = np.zeros((batch, trace_cap), dtype=np.int32) if trace_cap else None
        r = FiberResult()
        r.firstdz = _ptr(self.firstdz)
        r.ncycle = self.ncycle.ctypes.data_as(_ip)
        r.ntot = self.ntot.ctypes.data_as(_ip)
        r.status = self.status.ctypes.data_as(_ip)
        if trace_cap:
            r.trace_dz = _ptr(self.trace_dz)
            r.trace_ntrunk = self.trace_ntrunk.ctypes.data_as(_ip)
        r.trace_cap = trace_cap
        self.c = r

    def schedule(self, b=0):
        n = int(self.ncycle[b])
        return self.trace_dz[b, :n].copy(), self.trace_ntrunk[b, :n].copy()


def complex_field(x: np.ndarray, y):
    """Field struct over two complex128 arrays (PMX_COMPLEX); arrays must be C-contiguous
    [batch][nfc][nfft] and stay alive."""
    f = Field()
    f.layout = PMX_COMPLEX
    f.xr = x.ctypes.data_as(_dp)
    f.yr = y.ctypes.data_as(_dp) if y is not None else None
    return f


def planar_field(xr, xi, yr, yi):
    f = Field()
    f.layout = PMX_PLANAR
    f.xr, f.xi, f.yr, f.yi = _ptr(xr), _ptr(xi), _ptr(yr), _ptr(yi)
    return f


class DeviceField:
    """A field resident in HBM: [batch][nfc][nfft] two-polarization samples."""

    def __init__(self, ctx: Context, nfft, nfc=1, batch=1, precision=PMX_F64):
        self.ctx, self.nfft, self.nfc, self.batch = ctx, int(nfft), int(nfc), int(batch)
        self.precision = int(precision)
        h = C.c_void_p()
        ctx.check(ctx.lib.pmx_field_create(ctx.h, self.nfft, self.nfc, self.batch, precision, C.byref(h)))
        self.h = h

    def _as_cols(self, a, nb):
        # accept [nfft, nfc] (GSTATE layout) for nb == 1, or [nb, nfc, nfft]
        a = np.asarray(a, dtype=np.complex128)
        if a.ndim == 2 and nb == 1 and a.shape == (self.nfft, self.nfc):
            a = a.T[None]
        return np.ascontiguousarray(a.reshape(nb, self.nfc, self.nfft))

    def upload(self, x, y=None, b0=0, nb=None):
        nb = self.batch if nb is None else nb
        xs = self._as_cols(x, nb)
        ys = self._as_cols(y, nb) if y is not None else None
        f = complex_field(xs, ys)
        self.ctx.check(self.ctx.lib.pmx_field_upload(self.h, C.byref(f), b0, nb))
        self.ctx.sync()  # host arrays may be temporaries

    def download(self, b0=0, nb=None):
        """-> (x, y) complex128 arrays [nb, nfc, nfft]."""
        nb = self.batch if nb is None else nb
        x = np.empty((nb, self.nfc, self.nfft), dtype=np.complex128)
        y = np.empty_like(x)
        f = complex_field(x, y)
        self.ctx.check(self.ctx.lib.pmx_field_download(self.h, C.byref(f), b0, nb))
        return x, y

    def download_into(self, x: np.ndarray, y: np.ndarray, b0=0, nb=None):
        """D2H straight into caller-owned C-contiguous complex128 buffers of nb*nfc*nfft elements
        (keeps pinned buffers pinned)."""
        nb = self.batch if nb is None else nb
        for a in (x, y):
            if a.dtype != np.complex128 or not a.flags['C_CONTIGUOUS'] or a.size != nb * self.nfc * self.nfft:
                raise ValueError('download_into needs C-contiguous complex128 buffers of the field size')
        f = complex_field(x, y)
        self.ctx.check(self.ctx.lib.pmx_field_download(self.h, C.byref(f), b0, nb))

    def broadcast_from(self, src: 'DeviceField'):
        self.ctx.check(self.ctx.lib.pmx_field_broadcast(self.h, src.h))

    @property
    def device_ptr(self):
        return self.ctx.lib.pmx_field_device_ptr(self.h)

    def close(self):
        if getattr(self, 'h', None):
            self.ctx.lib.pmx_field_destroy(self.h)
            self.h = None

    def __del__(self):
        # at interpreter shutdown objects die in no particular order (a context before its plans): leave them to the process exit
        if sys.is_finalizing():
            return
        try:
            self.close()
        except Exception:
            pass


class Plan:
    def __init__(self, ctx: Context, desc: FiberDesc, keep):
        self.ctx, self.desc, self.keep = ctx, desc, keep
        h = C.c_void_p()
        ctx.check(ctx.lib.pmx_plan_create(ctx.h, C.byref(desc), C.byref(h)))
        self.h = h

    def set_plates(self, db0, theta, epsilon, plate_sets=1):
        a, b, c = _f64(db0).reshape(-1), _f64(theta).reshape(-1), _f64(epsilon).reshape(-1)
        self.ctx.check(self.ctx.lib.pmx_plan_set_plates(self.h, plate_sets, _ptr(a), _ptr(b), _ptr(c)))

    def set_length(self, length: float):
        """one-step (linear-flag) plans: the next execute applies lin_step(betat*length, u)"""
        self.ctx.check(self.ctx.lib.pmx_plan_set_length(self.h, float(length)))

    def execute(self, field: DeviceField, trace_cap=0) -> Result:
        res = Result(field.batch, trace_cap)
        self.ctx.check(self.ctx.lib.pmx_fiber_exec(self.h, field.h, C.byref(res.c)))
        return res

    def link_exec(self, field: DeviceField, link, keep) -> 'Result':
        """nspan x [fiber ; ampliflat] on the resident field (pmx_link_exec); -> Result with [nspan*batch] entries,
        span-major"""
        res = Result(field.batch * int(link.nspan))
        self.ctx.check(self.ctx.lib.pmx_link_exec(self.h, field.h, C.byref(link), C.byref(res.c)))
        return res

    def close(self):
        if getattr(self, 'h', None):
            self.ctx.lib.pmx_plan_destroy(self.h)
            self.h = None

    def __del__(self):
        # at interpreter shutdown objects die in no particular order (a context before its plans): leave them to the process exit
        if sys.is_finalizing():
            return
        try:
            self.close()
        except Exception:
            pass


class DbpPlan(Plan):
    """Digital backpropagation of a link (pmx_dbp_create): execute(field) runs it in place on a resident field.  With a
    band (DbpBand: shift, decim) it is the DBP of one channel of a one-column field at nfft/decim samples
    (pmx_dbp_channel_create)."""

    def __init__(self, ctx: Context, desc: FiberDesc, keep, dbp: DbpDesc, dbp_keep, band: 'DbpBand' = None):
        self.ctx, self.desc, self.keep, self.dbp, self.dbp_keep, self.band = ctx, desc, keep, dbp, dbp_keep, band
        h = C.c_void_p()
        if band is None:
            ctx.check(ctx.lib.pmx_dbp_create(ctx.h, C.byref(desc), C.byref(dbp), C.byref(h)))
        else:
            ctx.check(ctx.lib.pmx_dbp_channel_create(ctx.h, C.byref(desc), C.byref(dbp), C.byref(band), C.byref(h)))
        self.h = h

    def execute(self, field: DeviceField, trace_cap=0):
        self.ctx.check(self.ctx.lib.pmx_dbp_exec(self.h, field.h))

    def set_plates(self, db0, theta, epsilon, plate_sets=1):
        """the waveplates of a PMD-aware plan (pmx_dbp_set_plates): each [nspan][plate_sets][nplates] in forward span and
        plate order and sign, as the link took them; plate_sets is 1 or the batch"""
        a, b, c = _f64(db0).reshape(-1), _f64(theta).reshape(-1), _f64(epsilon).reshape(-1)
        n = int(self.dbp.nspan) * int(plate_sets) * int(self.desc.nplates)
        if not (a.size == b.size == c.size == n):
            raise ValueError('plates must be [nspan][plate_sets][nplates] = %d values each' % n)
        self.ctx.check(self.ctx.lib.pmx_dbp_set_plates(self.h, int(plate_sets), _ptr(a), _ptr(b), _ptr(c)))

    def set_filter(self, bw_bins):
        """filtered DBP (pmx_dbp_set_filter): a Gaussian low-pass of one-sided -3 dB bandwidth bw_bins, in DFT bins of the
        plan's grid, on the intensity of every nonlinear step; 0 switches it off"""
        self.ctx.check(self.ctx.lib.pmx_dbp_set_filter(self.h, float(bw_bins)))

    def set_taps(self, taps):
        """enhanced split-step DBP (pmx_dbp_set_taps): the real circular FIR taps c[0..2K] (c[K] at lag 0) on the intensity
        of every nonlinear step, on the plan's grid; None or [] switches them off"""
        a = check_taps(taps)
        self.ctx.check(self.ctx.lib.pmx_dbp_set_taps(self.h, int(a.size), _ptr(a) if a.size else None))


MAX_TAPS = 65


def check_taps(taps) -> np.ndarray:
    """-> the taps as a contiguous float64 vector (empty: no taps); ValueError with pmx_dbp_set_taps's message for what
    it refuses without a plan: an even count, more than MAX_TAPS, a non-finite tap"""
    a = np.ascontiguousarray(np.asarray([] if taps is None else taps, dtype=np.float64).ravel())
    if a.size > MAX_TAPS or (a.size and a.size % 2 == 0):
        raise ValueError('pmx_dbp_set_taps: ntaps must be odd and at most %d (0: no taps), got %d' % (MAX_TAPS, a.size))
    bad = np.flatnonzero(~np.isfinite(a))
    if bad.size:
        raise ValueError('pmx_dbp_set_taps: tap %d is not finite' % bad[0])
    return a


def make_band(shift, decim):
    """-> DbpBand: the channel brought to baseband by `shift` bins (pmx_field_modulate's m), backpropagated on nfft/decim
    samples"""
    b = DbpBand()
    b.shift, b.decim = int(shift), int(decim)
    return b


def make_dbp(nspan, gain=0.0, steps_per_span=None, step_len=None, span_steps=None, xi=1.0, pmd=False):
    """-> (DbpDesc, keep-alive dict).  Either steps_per_span (uniform steps) or step_len: the steps of one span in forward
    order (every span gets them), or with span_steps [nspan] the steps of all spans concatenated.  pmd: PMD-aware DBP
    (the plates follow with DbpPlan.set_plates)."""
    keep = {}
    d = DbpDesc()
    d.nspan, d.xi, d.gain, d.pmd = int(nspan), float(xi), float(gain), int(bool(pmd))
    if step_len is None:
        d.steps_per_span = int(1 if steps_per_span is None else steps_per_span)
        return d, keep
    if steps_per_span is not None:
        raise ValueError('give steps_per_span or step_len, not both')
    keep['step_len'] = _f64(np.asarray(step_len, dtype=np.float64).reshape(-1))
    if span_steps is None:
        keep['step_len'] = np.ascontiguousarray(np.tile(keep['step_len'], int(nspan)))
        span_steps = [keep['step_len'].size // int(nspan)] * int(nspan)
    keep['span_steps'] = np.ascontiguousarray(np.asarray(span_steps, dtype=np.int32).reshape(-1))
    if keep['span_steps'].size != int(nspan):
        raise ValueError('span_steps must give the steps of every span')
    if int(keep['span_steps'].astype(np.int64).sum()) != keep['step_len'].size:
        raise ValueError('step_len must hold sum(span_steps) steps')
    d.steps_per_span = 0
    d.step_len = _ptr(keep['step_len'])
    d.span_steps = keep['span_steps'].ctypes.data_as(_ip)
    return d, keep


class Filter(Plan):
    """u <- ifft(fft(u) .* H) on a device field (pmx_filter_create).  H: [nfft] or [nfft, nfc] complex, in the order of
    GSTATE.FN; one column filters every field column alike."""

    def __init__(self, ctx: Context, nfft, nfc, H, batch=1, precision=PMX_F64):
        hh = np.asarray(H, dtype=np.complex128)
        hh = hh.reshape(nfft, -1) if hh.ndim > 1 else hh.reshape(nfft, 1)
        if hh.shape[1] not in (1, nfc):
            raise ValueError('H must have one column, or one per field column')
        self.ctx, self.desc, self.keep = ctx, None, None
        hc = np.ascontiguousarray(hh.T)                       # [hcols][nfft]
        h = C.c_void_p()
        ctx.check(ctx.lib.pmx_filter_create(ctx.h, int(nfft), int(nfc), int(batch), int(precision),
                                            hc.ctypes.data_as(_dp), hc.shape[0], C.byref(h)))
        self.h = h


def make_link(nspan, gain=0.0, sigma=None, plates=None, plate_sets=1, noise=None, seeds=None, first=0, asepol=3):
    """-> (LinkDesc, keep-alive dict).  plates: (db0, theta, epsilon) each [nspan][plate_sets][nplates] or None;
    noise: [nspan][batch][2*nfc][nfft] complex128 or None; seeds: [nspan] ints or None."""
    keep = {}
    l = LinkDesc()
    l.nspan, l.plate_sets, l.gain = int(nspan), int(plate_sets), float(gain)
    l.realization0 = int(first)          # global index of the batch's first realization (ASE generator key)
    l.asepol = int(asepol)               # 1: ASE on X only, 2: on Y only, 3: both (options.onepol)
    if plates is not None:
        for name, a in zip(('db0', 'theta', 'epsilon'), plates):
            keep[name] = _f64(a).reshape(-1)
            if keep[name].size % int(nspan):
                raise ValueError('plates must hold nspan draws')
            setattr(l, name, _ptr(keep[name]))
    if sigma is not None:
        keep['sigma'] = _f64(np.atleast_1d(sigma))
        l.sigma = _ptr(keep['sigma'])
    if noise is not None:
        keep['noise'] = np.ascontiguousarray(noise, dtype=np.complex128)
        l.noise = keep['noise'].ctypes.data_as(_dp)
    if seeds is not None:
        keep['seeds'] = np.ascontiguousarray(seeds, dtype=np.uint64)
        if keep['seeds'].size != int(nspan):
            raise ValueError('one ASE seed per span')
        l.seeds = keep['seeds'].ctypes.data_as(C.POINTER(C.c_uint64))
    return l, keep


def field_mux(ctx: Context, field: DeviceField, sigx, sigy, ndfn, scale=None, delayx=None, delayy=None):
    """create_field('unique') on the device (pmx_field_mux): sigx/sigy [nfft, nch] complex (GSTATE layout)."""
    nch = int(np.shape(sigx)[1])
    xs = np.ascontiguousarray(np.asarray(sigx, dtype=np.complex128).T)          # [nch][nfft]
    ys = np.ascontiguousarray(np.asarray(sigy, dtype=np.complex128).T) if sigy is not None else None
    f = complex_field(xs, ys)
    i64 = C.POINTER(C.c_int64)
    nd = np.ascontiguousarray(ndfn, dtype=np.int64)
    sc = _f64(scale) if scale is not None else None
    dx = np.ascontiguousarray(delayx, dtype=np.int64) if delayx is not None else None
    dy = np.ascontiguousarray(delayy, dtype=np.int64) if delayy is not None else None
    ctx.check(ctx.lib.pmx_field_mux(field.h, C.byref(f), nch, nd.ctypes.data_as(i64), _ptr(sc),
                                    dx.ctypes.data_as(i64) if dx is not None else None,
                                    dy.ctypes.data_as(i64) if dy is not None else None))


def scalar_nl_exec(ctx: Context, field: DeviceField, gam, leff: float, atten: float, spm: bool, xpm: bool):
    """nl_step (fiber.m:786-803) followed by the attenuation factor of the same sub-step"""
    g = _f64(np.atleast_1d(gam))
    ctx.check(ctx.lib.pmx_scalar_nl_exec(ctx.h, field.h, _ptr(g), float(leff), float(atten), int(bool(spm)), int(bool(xpm))))


def field_max_power(ctx: Context, field: DeviceField) -> np.ndarray:
    """max_n |ux|^2 + |uy|^2 per realization and column -> [batch, nfc] (nextstep's Umax, fiber.m:693-698)"""
    out = np.zeros(field.batch * field.nfc)
    ctx.check(ctx.lib.pmx_field_max_power(ctx.h, field.h, _ptr(out)))
    return out.reshape(field.batch, field.nfc)


def field_maxdiff2(ctx: Context, a: DeviceField, b: DeviceField) -> float:
    out = np.zeros(1)
    ctx.check(ctx.lib.pmx_field_maxdiff2(ctx.h, a.h, b.h, _ptr(out)))
    return float(out[0])


def field_lincomb(ctx: Context, dst: DeviceField, ca: float, a: DeviceField, cb: float, b: DeviceField):
    """dst <- ca*a - cb*b"""
    ctx.check(ctx.lib.pmx_field_lincomb(ctx.h, dst.h, float(ca), a.h, float(cb), b.h))


def ampliflat_exec(ctx: Context, field: DeviceField, gain: float, sigma, noise=None, seed=0, asepol=3):
    """asepol: 1 = ASE on X only, 2 = on Y only, 3 = both (options.onepol, ampliflat.m:107-118)"""
    s = _f64(np.atleast_1d(sigma))
    n = None
    if noise is not None:
        n = np.ascontiguousarray(noise, dtype=np.complex128)
    ctx.check(ctx.lib.pmx_ampliflat_exec_pol(ctx.h, field.h, float(gain), _ptr(s),
                                             n.ctypes.data_as(_dp) if n is not None else None,
                                             C.c_uint64(int(seed)), int(asepol)))
    if n is not None:
        ctx.sync()


def qpsk_count(ctx: Context, field: DeviceField, sym, nsymb: int, nt: int, counts_dev_ptr: int):
    """Error counts of every realization of `field` into a device int64 buffer (pmx_qpsk_count)."""
    s = np.ascontiguousarray(sym, dtype=np.uint8).reshape(2, nsymb)
    ctx.check(ctx.lib.pmx_qpsk_count(ctx.h, field.h, s.ctypes.data_as(C.c_void_p), int(nsymb), int(nt),
                                     C.c_void_p(int(counts_dev_ptr))))
