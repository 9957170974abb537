"""B200-native solver for the reference's one data-parallel hot path: fixed-step RK4 over the
Yaman/Agrawal coupled-amplitude FWM system, batched over parameter sweeps.

The submodules keep the reference's module and function names (config, constants,
frequency_plan, dispersion, phase_matching, parameters, integrators, yaman_model, simulation,
scan_mismtach, io_fwm) so callers switch by changing the import; `nwave` is the N-wave
generalisation and `small_signal` the host-side algebra on small-signal transfer matrices.  All arithmetic of the path runs in libfpa_b200.so (CUDA, sm_100a) behind the
C ABI of include/fpa_b200.h; there is no CPU fallback.
"""
from . import _lib, _device  # noqa: F401
from . import (config, constants, dispersion, frequency_plan, integrators, io_fwm,  # noqa: F401
               nwave, parameters, phase_matching, scan_mismtach, sharding, simulation, small_signal,
               yaman_model)

__all__ = ["config", "constants", "dispersion", "frequency_plan", "integrators", "io_fwm", "nwave",
           "parameters", "phase_matching", "scan_mismtach", "sharding", "simulation", "small_signal", "yaman_model"]
