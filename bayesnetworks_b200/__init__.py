"""bayesnetworks_b200 -- B200 (sm_100a) implementation of the structure-MCMC scoring
hot path of USCbiostats/bayesnetworks, behind the reference's own interface.

    from bayesnetworks_b200 import bn_mcmc, create_network
    out = bn_mcmc(X, graph, N=50000)      # columns iter, ChangedNode, movetype, globalLL, ...

All compute runs in ``libbn_b200.so`` (hand-written CUDA, C ABI in include/bn_b200.h).
"""
from .network import Network, create_network, read_dag, read_data  # noqa: F401
from .api import (BestGraph, ChainResult, ChainState, Context, TRACE_COLUMNS, bn_mcmc, main_fun,  # noqa: F401
                  set_default_stream)
from ._lib import BnError  # noqa: F401
from .summary import ancestor_posterior, best_graph, summarize, summarize_result  # noqa: F401

__all__ = ["Network", "create_network", "read_dag", "read_data", "Context", "ChainResult", "ChainState",
           "TRACE_COLUMNS", "bn_mcmc", "main_fun", "BnError", "summarize", "summarize_result",
           "ancestor_posterior", "BestGraph", "best_graph"]
