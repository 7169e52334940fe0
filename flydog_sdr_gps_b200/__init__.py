"""B200-native GNSS acquisition engine: the FFT parallel-code-phase search of gps/search.cpp as
hand-written sm_100a CUDA kernels behind a C ABI (include/acq_b200.h)."""
from . import sats  # noqa: F401
from .engine import (AcqEngine, AcqError, BIN_HZ, BLOCK_BYTES, CELL_DTYPE, FINE_DTYPE, LAGS_E1B, LAGS_L1, N,  # noqa: F401
                     PEAK2_DTYPE, RECORD_DTYPE, WRAP_CIRCULAR, WRAP_REFERENCE, default_params, microbench)
