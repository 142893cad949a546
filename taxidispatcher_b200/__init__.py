"""taxidispatcher_b200 -- B200-native (sm_100a) drop-in for the taxidispatcher dispatch hot path:
cost-matrix build -> exact balanced assignment -> LCM greedy -> 2..4-passenger pool finder.

    from taxidispatcher_b200 import calculate_cost, solve, LCM, find_pool

The compute surface lives in .dispatch and needs the in-tree CUDA library
(taxidispatcher_b200/libtaxidispatch.so, built by taxidispatcher_b200.build) and a CUDA device;
there is no CPU fallback.  Importing this package alone touches neither.
"""
__version__ = "0.1.0"

_DISPATCH = ("BIG_COST", "Engine", "engine", "calculate_cost", "solve", "solve_dispatch", "solve_full", "LCM",
             "LCM_heuristic", "LCM_split", "LCM_greedy_opt", "LCM_simulate", "LCM_java", "find_pool", "find_pool_all", "find_pool_block", "find_pool_pairs",
             "find_pool_pairs_batch", "find_pool_pairs_exact", "find_pool_pairs_exact_batch", "find_pool_all_batch",
             "pool_merge", "pack_batch", "solve_stands_batch", "solve_assignment_stands", "solve_batch", "LCM_batch", "TaxiDispatchError")


def __getattr__(name):
    if name in _DISPATCH:
        from . import dispatch
        return getattr(dispatch, name)
    raise AttributeError(name)
