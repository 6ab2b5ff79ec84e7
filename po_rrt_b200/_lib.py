"""ctypes loader for libporrt_b200.so (the C ABI declared in include/porrt_b200.h).

There is no CPU fallback: if the shared library is missing this raises, and every entry point fails with
PORRT_ERR_CUDA when no sm_100 device is present.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PORRT_B200_LIB") or os.path.join(_HERE, "libporrt_b200.so")  # override: A/B builds of the kernels

vp, i32, i64, f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_double
pp = C.POINTER

# name -> (restype, argtypes); mirrors include/porrt_b200.h one to one
SIGNATURES = {
    "porrt_version": (C.c_char_p, []),
    "porrt_pgm_read": (i32, [vp, C.c_char_p, vp, i64, vp, vp]),
    "porrt_pgm_write": (i32, [vp, C.c_char_p, vp, i32, i32, i32]),
    "porrt_graph_load_json": (i32, [vp, C.c_char_p, vp]),
    "porrt_graph_info": (i32, [vp, vp, vp, vp, vp, vp]),
    "porrt_graph_arrays": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "porrt_graph_destroy": (i32, [vp]),
    "porrt_graph_save_json": (i32, [vp, C.c_char_p, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32]),
    "porrt_ctx_create": (i32, [i32, pp(vp)]),
    "porrt_ctx_destroy": (i32, [vp]),
    "porrt_ctx_set_stream": (i32, [vp, vp]),
    "porrt_ctx_synchronize": (i32, [vp]),
    "porrt_ctx_bind_host_thread": (i32, [vp, pp(i32)]),
    "porrt_last_error": (C.c_char_p, [vp]),
    "porrt_ctx_launch_count": (i64, [vp]),
    "porrt_ctx_last_phase_ms": (i32, [vp, vp, i32, pp(i32)]),
    "porrt_measure_l2_gather": (i32, [vp, i64, pp(f64)]),
    "porrt_map_upload": (i32, [vp, vp, vp, i32, i32, vp, vp, i32, f64]),
    "porrt_map_info": (i32, [vp, pp(i32), pp(i32), pp(i32), pp(i32)]),
    "porrt_map_zone_positions": (i32, [vp, vp]),
    "porrt_map_world_validities": (i32, [vp, vp]),
    "porrt_state_validity": (i32, [vp, vp, i64, vp]),
    "porrt_edge_validity": (i32, [vp, vp, vp, i64, vp, vp]),
    "porrt_visibility": (i32, [vp, vp, i64, vp, vp]),
    "porrt_edge_validity_indexed": (i32, [vp, vp, vp, i64, vp, vp]),
    "porrt_edge_validity_i8": (i32, [vp, vp, vp, i64, vp]),
    "porrt_edge_validity_indexed_i8": (i32, [vp, vp, vp, i64, vp]),
    "porrt_edge_validity_csr_i8": (i32, [vp, vp, vp, i64, i32, vp]),
    "porrt_ctx_set_option": (i32, [vp, i32, i64]),
    "porrt_state_validity_dev": (i32, [vp, vp, i64, vp]),
    "porrt_edge_validity_dev": (i32, [vp, vp, vp, i64, vp, vp]),
    "porrt_visibility_dev": (i32, [vp, vp, i64, vp, vp]),
    "porrt_transition_valid": (i32, [vp, vp, vp, i64, vp, vp, vp]),
    "porrt_partial_shortcut": (i32, [vp, vp, i32, vp, i32, C.c_uint64, pp(i32), pp(i32)]),
    "porrt_partial_shortcut_batch": (i32, [vp, vp, vp, i32, vp, i32, C.c_uint64, vp, pp(i32)]),
    "porrt_vertices_set": (i32, [vp, vp, i64, f64]),
    "porrt_vertices_append": (i32, [vp, vp, i64]),
    "porrt_vertices_set_dev": (i32, [vp, vp, i64, f64, vp, vp]),
    "porrt_vertices_count": (i32, [vp, pp(i64)]),
    "porrt_radius_query": (i32, [vp, vp, vp, i64, vp, vp, i32, vp, vp, vp, i64, pp(i64)]),
    "porrt_nearest": (i32, [vp, vp, i64, vp, i32, vp, vp, vp, vp]),
    "porrt_knn": (i32, [vp, vp, i64, i32, vp, vp]),
    "porrt_kd_preorder_rank": (i32, [vp, vp, i64, vp]),
    "porrt_prm_build": (i32, [vp, vp, i64, f64, f64, vp, vp, i64, pp(i64), vp]),
    "porrt_prm_fetch": (i32, [vp, vp, vp, i64]),
    "porrt_sssp_worlds_prm": (i32, [vp, vp, vp, vp, pp(i32)]),
    "porrt_prm_plan_paths": (i32, [vp, vp, vp, i64, vp, vp, vp, vp, vp, vp, i64, pp(i64)]),
    "porrt_sssp_worlds": (i32, [vp, i64, vp, vp, vp, vp, vp, i32, i32, i32, vp, vp, vp, pp(i32)]),
    "porrt_policy_decompose": (i32, [vp, i64, vp, vp, vp, vp, i32, pp(i32)]),
    "porrt_policy_expected_cost": (i32, [vp, vp, vp, i64, vp, i32, i32, pp(f64)]),
    "porrt_refine_policy_reparent": (i32, [vp, vp, vp, vp, i64, f64, vp, vp, vp, vp, vp, i64, vp, vp, vp, vp]),
    "porrt_refine_policy_shortcut": (i32, [vp, vp, vp, vp, i64, i32, C.c_uint64, vp, vp, vp, vp, vp, i64, vp, vp, vp]),
    "porrt_belief_result": (i32, [vp, vp, vp, vp, vp]),
    "porrt_belief_vi": (i32, [vp, i64, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, i32, vp, vp, vp, i32, vp, vp, pp(i32), vp]),
    "porrt_extract_policy": (i32, [vp, vp, vp, vp, vp, i64, pp(i64), pp(f64)]),
    "porrt_conditional_dijkstra": (i32, [vp, i64, vp, vp, vp, vp, vp, vp, i32, i32, vp, i32, vp, pp(i32)]),
    "porrt_extract_policy_graph": (i32, [vp, i64, vp, vp, vp, vp, vp, vp, i32, i32, vp, vp, vp, vp, i64, pp(i64), pp(f64)]),
    "porrt_conditional_dijkstra_nd": (i32, [vp, i32, i64, vp, vp, vp, vp, vp, vp, i32, i32, vp, i32, vp, pp(i32)]),
    "porrt_extract_policy_graph_nd": (i32, [vp, i32, i64, vp, vp, vp, vp, vp, vp, i32, i32, vp, vp, vp, vp, i64, pp(i64), pp(f64)]),
    "porrt_mmprm_plan": (i32, [vp, i32, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, pp(i64), pp(i32), vp]),
    "porrt_mmprm_fetch_graph": (i32, [vp, vp, vp, i64, vp, vp]),
    "porrt_qmdp_react": (i32, [vp, i64, vp, vp, vp, i32, vp, i64, vp, i32, f64, vp, vp, i64, pp(i64), pp(i64)]),
    "porrt_heuristic_radius": (i32, [i64, f64, f64, i32, pp(f64)]),
    "porrt_steer": (i32, [vp, vp, i64, f64]),
    "porrt_steer_nd": (i32, [vp, vp, i64, i32, f64]),
    "porrt_sampler_create": (i32, [C.c_uint64, pp(vp)]),
    "porrt_sampler_destroy": (i32, [vp]),
    "porrt_sampler_continuous": (i32, [vp, vp, vp, i32, i64, vp]),
    "porrt_sampler_discrete": (i32, [vp, C.c_uint64, i64, vp]),
    "porrt_square_goal": (i32, [vp, i32, f64, vp, i64, vp]),
    "porrt_square_goal_examples": (i32, [vp, vp, i32, i32, vp]),
    "porrt_reach_create": (i32, [i32, vp, pp(vp)]),
    "porrt_reach_destroy": (i32, [vp]),
    "porrt_reach_add_node": (i32, [vp, vp]),
    "porrt_reach_add_final_node": (i32, [vp, i64, vp]),
    "porrt_reach_add_edge": (i32, [vp, i64, i64, vp]),
    "porrt_reach_count": (i32, [vp, pp(i64), pp(i32)]),
    "porrt_reach_masks": (i32, [vp, i64, i64, vp]),
    "porrt_reach_final_nodes_for_world": (i32, [vp, i32, vp, i64, pp(i64)]),
    "porrt_reach_finals": (i32, [vp, vp, vp, i64, pp(i64)]),
    "porrt_reach_is_final_set_complete": (i32, [vp, pp(i32)]),
    "porrt_reachable_belief_states": (i32, [vp, vp, vp, i32, pp(i32)]),
    "porrt_pto_grow": (i32, [vp, vp, vp, vp, C.c_uint64, vp, vp, i32, f64, f64, f64, i64, i64, vp, pp(i32), pp(i32), vp]),
    "porrt_pto_fetch": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "porrt_pto_grow_batch": (i32, [vp, i32, vp, vp, vp, vp, vp, vp, i32, f64, f64, f64, i64, i64, vp, vp, vp, vp]),
    "porrt_pto_fetch_roadmap": (i32, [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp]),
    "porrt_pto_plan_batch": (i32, [vp, vp, i32, i32, vp, vp, vp, vp, vp, vp, vp, i64, pp(i64), vp, vp]),
    "porrt_rrt_grow_batch": (i32, [vp, i32, vp, vp, vp, vp, vp, vp, i32, f64, f64, f64, i64, i64, vp, vp, vp, vp]),
    "porrt_rrt_grow": (i32, [vp, C.c_uint64, vp, vp, vp, vp, vp, i32, f64, f64, f64, i64, i64, vp, pp(i32), pp(i32), vp]),
    "porrt_rrt_fetch_tree": (i32, [vp, i32, vp, vp, vp, vp]),
    "porrt_rrt_grow_queries": (i32, [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, f64, f64, i64, i64, vp, vp, vp, vp]),
    "porrt_rrt_best_paths": (i32, [vp, vp, vp, vp, vp, i64, pp(i64)]),
    "porrt_comm_unique_id": (i32, [vp]),
    "porrt_comm_init": (i32, [vp, vp, i32, i32]),
    "porrt_comm_destroy": (i32, [vp]),
    "porrt_comm_info": (i32, [vp, pp(i32), pp(i32), pp(i32)]),
    "porrt_shard_range": (i32, [i64, i32, i32, pp(i64), pp(i64)]),
    "porrt_comm_all_gather_dev": (i32, [vp, vp, vp, i64, i64]),
    "porrt_comm_all_gatherv_dev": (i32, [vp, vp, vp, vp]),
}

_lib = None


def load():
    """Load the shared library and type every exported symbol; raises if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libporrt_b200.so not built (run `python -c 'import __graft_entry__ as g; g.build()'` or "
                "`make -C po_rrt_b200/csrc`); po_rrt_b200 has no CPU fallback")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib
