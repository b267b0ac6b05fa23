"""polmux_b200: the Optilux/Polmux split-step Fourier fiber channel on NVIDIA B200.

One hot path, B200-native: ``fiber(x, flag)`` with the reference's call signature
and GSTATE field layout, backed by a C-ABI CUDA library (include/polmux_ssfm.h).
"""
from .gstate import CONSTANTS, GSTATE, reset_all, seed  # noqa: F401
from .field import create_field  # noqa: F401
from .fiber import fiber, fiber_setup, LAST as FIBER_LAST  # noqa: F401
from .ampliflat import ampliflat  # noqa: F401
from .inverse_pmd import inverse_pmd  # noqa: F401
from .link import link  # noqa: F401
from .dbp import dbp  # noqa: F401
from .receiver import receiver_cohmix, myfilter, evaldelay  # noqa: F401
from .dsp import dsp4cohdec  # noqa: F401
from ._lib import PolmuxError, Context, DeviceField, Plan  # noqa: F401

__version__ = '0.1.0'
