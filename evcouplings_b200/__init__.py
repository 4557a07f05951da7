"""
evcouplings_b200 -- B200-native pseudo-likelihood Potts-model inference engine that drops in
behind ``evcouplings.couplings.protocol.standard`` (replaces the external plmc binary).

    import evcouplings.couplings.tools as ct, evcouplings_b200
    ct.run_plmc = evcouplings_b200.run_plmc

Python host code (this package) -> ctypes -> csrc/libevcplm.so (hand-written sm_100a CUDA).
There is no CPU execution path.
"""
from .tools import run_plmc, parse_plmc_log, PlmcResult          # noqa: F401
from ._lib import EngineUnavailableError, EngineError             # noqa: F401
from .mean_field import MeanFieldDCA, MeanFieldModel, run_mean_field  # noqa: F401

__version__ = "0.1.0"


def install_into_reference():
    """Monkey-patch the reference package so that its couplings protocols use this engine."""
    import evcouplings.couplings.tools as ct
    ct.run_plmc = run_plmc
    return ct


def install_mean_field_into_reference():
    """Monkey-patch the reference's couplings protocol so that its ``mean_field`` protocol uses this engine."""
    import evcouplings.couplings.protocol as cp
    cp.MeanFieldDCA = MeanFieldDCA
    return cp
