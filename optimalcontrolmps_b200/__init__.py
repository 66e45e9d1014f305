"""optimalcontrolmps_b200 -- B200-native (sm_100a) engine for the hot path of fskovbo/OptimalControlMPS.

The package holds the CUDA sources of ``libocmps.so`` (``csrc/``), its ctypes binding (``_lib``) and a
host-side mirror of the reference's C++ interface (``api``).  It never falls back to the CPU.
"""
import os as _os

# The engine fills the GPU with independent chains (psi / xi sweeps, batched controls, Hessian rows), one CUDA stream
# (plus a side stream) each.  Streams are multiplexed onto CUDA_DEVICE_MAX_CONNECTIONS hardware queues, 8 by default:
# with more streams than queues unrelated chains serialise behind each other (measured: the rows of a sharded Hessian take
# 4.0 s with 8 queues and 2.1 s with 32).  The variable is read when the CUDA context is created, so it has to be set
# before anything in the process touches CUDA; a value the user has set is left alone.
_os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

from .api import (Args, BH_tDMRG, InitializeState, InitializeStateDMRG, BoseHubbard, Context, ControlBasis, ControlBasisFactory, DeviceMPS, IQMPS,
                  OptimalControl, SeedGenerator, SliceStore, batch_cost_gradient, energy, overlapC, overlapC_K, site_operator)
from ._lib import OcmpsError, LIB_PATH

__all__ = ["Args", "BH_tDMRG", "InitializeState", "InitializeStateDMRG", "BoseHubbard", "Context", "ControlBasis", "ControlBasisFactory", "DeviceMPS", "IQMPS",
           "OptimalControl", "SeedGenerator", "batch_cost_gradient", "energy", "SliceStore", "overlapC", "overlapC_K", "site_operator", "OcmpsError", "LIB_PATH"]
