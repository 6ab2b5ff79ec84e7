"""po_rrt_b200 -- B200 (sm_100a) implementation of po-rrt's data-parallel planning inner loop.

The product is po_rrt_b200/libporrt_b200.so (C ABI: include/porrt_b200.h, sources: po_rrt_b200/csrc/*.cu);
this package is the thin host-side mirror of the reference's interface used by tests and bench.py.
There is no CPU fallback: importing works anywhere, creating a Context needs the built library and a B200.
"""
from .api import (DOOR, SHELF, INVALID, PANIC_OOB, PANIC_ZONE_UNWRAP, PANIC_MULTI_ZONE, NODE_ACTION, NODE_OBSERVATION,
                  NODE_UNKNOWN, OPT_FORCE_LARGE_MAP_PATH, OPT_FORCE_GLOBAL_SWEEPS, OPT_FORCE_THREAD_PER_QUERY_NN, OPT_PRM_PATHS_CHUNK_COLUMNS, OPT_REPARENT_BRUTE_MAX_NODES,
                  PATH_FOUND, PATH_NONE, PATH_CYCLE, BeliefGraph, Context, KdTree, Map, MapShelfDomain, PRM, PTO, PTOBatch, RRT, RRTBatch, PorrtError, Reachability, Sampler, SquareGoal, dijkstra_worlds, dijkstra_worlds_resident_prm, heuristic_radius, mmprm_plan,
                  plan_belief_space, refine_policy_shortcut, refine_policy_reparent, policy_decompose, policy_expected_cost, react_qmdp, steer, words_from_bits)
from . import synth

__all__ = ["BeliefGraph", "Context", "Map", "MapShelfDomain", "KdTree", "PRM", "PTO", "PTOBatch", "RRT", "RRTBatch", "PorrtError", "dijkstra_worlds", "mmprm_plan", "plan_belief_space",
           "words_from_bits", "synth", "Reachability", "Sampler", "SquareGoal", "heuristic_radius", "react_qmdp", "steer"]
