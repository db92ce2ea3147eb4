"""bpl_next_b200 -- B200-native Dixon-Coles inference hot path for bpl-next.

The numbers come from hand-written sm_100a CUDA kernels behind the C ABI of ``include/bplx.h``
(``lib/libbplx.so``); there is no CPU fallback.  See DESIGN.md and INTEGRATION.md.
"""
from . import _abi, data  # noqa: F401

__version__ = "0.1.0"


def __getattr__(name):  # lazy: importing torch is slow and not needed for host-only users
    if name in ("Problem", "score_grid", "score_grid_host", "pointwise_loglik", "psis_loo",
                "simulate_table", "simulate_tournament", "posterior_predictive"):
        from . import problem
        return getattr(problem, name)
    if name in ("DixonColesMatchPredictor", "ExtendedDixonColesMatchPredictor", "NeutralDixonColesMatchPredictor",
                "NeutralDixonColesMatchPredictorWC",  # the four classes bpl/__init__.py:4-7 exports
                "DynamicNeutralDixonColesMatchPredictor"):  # not exported by the reference; fit only (SURVEY D3)
        from . import predictors
        return getattr(predictors, name)
    raise AttributeError(name)
