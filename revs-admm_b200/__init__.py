"""revs-admm_b200: the REVS distributed EV-charging ADMM loop, B200-native.

Host side mirrors the reference's modules (extract, lpsolver, revs_fixture); the numerical
path is hand-written CUDA for sm_100a behind the C ABI of include/revs_admm.h
(librevs_admm.so in this directory).  Import name: ``revs_admm_b200``.
"""
from . import _cabi, extract, feeder, lpsolver, revs_fixture  # noqa: F401
from ._cabi import (REVS_NET_CENTRAL, REVS_NET_ESTIMATE, REVS_NET_HOST, REVS_NET_REPAIRED, REVS_NET_SCHEDULE,  # noqa: F401
                    REVS_REL_DROP, REVS_REL_FLOW, REVS_REL_VOLTAGE, NetworkSummary, RevsError, Solver, contract, device_count,
                    central_status, expand_schedule, hosting_totals, screen_contract)
from .parallel import PipelinedSolver  # noqa: F401
from .revs_fixture import REVS  # noqa: F401

__version__ = "0.1.0"
