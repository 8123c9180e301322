"""basevar_b200: B200-native (sm_100a) implementation of the `basevar basetype` per-site statistical core.

The product is the CUDA library ``libbasevar_b200.so`` behind the C ABI of ``include/basevar_b200.h``;
this package is its thin Python host layer (ctypes).  There is no CPU fallback anywhere in here.
"""
from . import capi, synth  # noqa: F401
from .capi import BvError, SITE_OUT_DTYPE, cli_min_af  # noqa: F401
from .engine import (BaseTypeEngine, DeviceResult, dense_to_sparse, device_to_numpy, sparse_encode16, synth_fill_host,  # noqa: F401
                     synth_fill_rpr_host, synth_fill_sparse_host)

__version__ = "0.1.0"
