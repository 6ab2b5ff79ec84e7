//! pto_b200.rs -- planner-level swap for `PTO::plan_belief_space` (pto.rs:152-182): child module of `pto`
//! (`#[cfg(feature = "b200")] #[path = "pto_b200.rs"] mod b200;`), so it may fill the private `expected_costs_to_goals`.
//!
//! `build_belief_graph` (pto.rs:185-259) materialises V x B belief nodes and calls `observe` V x B times; with the feature on the
//! belief graph stays IMPLICIT on the device (belief node id = node * B + belief, node types and observation edges from
//! per-visible-zone-set tables, DESIGN.md 3.3): reachable beliefs + one visibility test per NODE + `porrt_belief_vi`, then the
//! policy walk `porrt_extract_policy` (belief_graph.rs:184-267).  Expected costs are bit-identical to conditional_dijkstra's.
//! Roadmap growth (`PTO::grow_graph`, pto.rs:55-139) has its swap too: `grow_graph_b200` runs the whole loop in ONE
//! `porrt_pto_grow` (speculative windows with an exact in-order commit, DESIGN.md 3.8) and copies the roadmap, the reachability
//! masks and the final nodes back into the planner's own structures, bit for bit what `grow_graph` builds; `grow_graphs_b200`
//! grows one planner per seed in ONE `porrt_pto_grow_batch` (the roadmaps share each window's launches, DESIGN.md 3.8).
#![cfg(feature = "b200")]

use super::PTO;
use crate::b200::{mask_from_words, words_from_mask, B200Domain};
use crate::b200_ffi::*;
use crate::common::*;
use crate::pto_graph::PTOFuncs;
use crate::qmdp_policy_extractor::b200::export_csr;

impl<'a> PTO<'a, B200Domain<'a>, 2> {
    /// PTO::grow_graph (pto.rs:55-139) on the device.  The samplers are PTO::new's (seed 0); the goal is a SquareGoal given as its
    /// (state, world mask) pairs.  Panics where the reference panics, returns Err where it does (pto.rs:131-138).
    pub fn grow_graph_b200(&mut self, start: &[f64; 2], goals: &[([f64; 2], WorldMask)], goal_max_dist: f64, max_step: f64,
                           search_radius: f64, n_iter_min: usize, n_iter_max: usize) -> Result<(), &'static str> {
        let ctx = self.fns.ctx;
        let mw = self.fns.mask_words();
        let goals_xy: Vec<f64> = goals.iter().flat_map(|(s, _)| s.iter().copied()).collect();
        let goal_masks: Vec<u64> = goals.iter().flat_map(|(_, m)| words_from_mask(m, mw)).collect();
        let (low, up) = (self.continuous_sampler.low, self.continuous_sampler.up);
        let (mut sizes, mut counters) = ([0i64; 4], [0i64; 4]);
        let (mut complete, mut panic_code) = (0i32, 0i32);
        let rc = unsafe {
            porrt_pto_grow(ctx.raw(), start.as_ptr(), low.as_ptr(), up.as_ptr(), 0, goals_xy.as_ptr(), goal_masks.as_ptr(),
                           goals.len() as i32, goal_max_dist, max_step, search_radius, n_iter_min as i64, n_iter_max as i64,
                           sizes.as_mut_ptr(), &mut complete, &mut panic_code, counters.as_mut_ptr())
        };
        ctx.check(rc); // PORRT_ERR_PANIC -> the reference's panic, with the library's message
        self.copy_back_b200(0, &sizes);
        if complete != 0 { Ok(()) } else { Err("final nodes are not reached for each world") }
    }

    /// PTO::grow_graph for one planner per seed in `seeds`, all grown in ONE `porrt_pto_grow_batch` call on this planner's map:
    /// planner r is `PTO::new(self.fns)` with both samplers seeded `seeds[r]`, filled with the roadmap, reachability and final
    /// nodes `grow_graph` builds with that seed.  Start, goal and parameters as `grow_graph_b200`.  A panic in one roadmap panics
    /// here with its code once the batch has been grown; Err where `grow_graph` returns Err (pto.rs:131-138).
    pub fn grow_graphs_b200(&self, seeds: &[u64], start: &[f64; 2], goals: &[([f64; 2], WorldMask)], goal_max_dist: f64,
                            max_step: f64, search_radius: f64, n_iter_min: usize, n_iter_max: usize)
                            -> Vec<(Self, Result<(), &'static str>)> {
        let ctx = self.fns.ctx;
        let mw = self.fns.mask_words();
        let n = seeds.len();
        let goals_xy: Vec<f64> = goals.iter().flat_map(|(s, _)| s.iter().copied()).collect();
        let goal_masks: Vec<u64> = goals.iter().flat_map(|(_, m)| words_from_mask(m, mw)).collect();
        let (low, up) = (self.continuous_sampler.low, self.continuous_sampler.up);
        let (mut sizes, mut counters) = (vec![0i64; 4 * n], vec![0i64; 4 * n]);
        let (mut status, mut panic_code) = (vec![0i32; n], vec![0i32; n]);
        ctx.check(unsafe {
            porrt_pto_grow_batch(ctx.raw(), n as i32, seeds.as_ptr(), start.as_ptr(), low.as_ptr(), up.as_ptr(), goals_xy.as_ptr(),
                                 goal_masks.as_ptr(), goals.len() as i32, goal_max_dist, max_step, search_radius, n_iter_min as i64,
                                 n_iter_max as i64, sizes.as_mut_ptr(), status.as_mut_ptr(), panic_code.as_mut_ptr(),
                                 counters.as_mut_ptr())
        });
        for r in 0..n {
            assert!(status[r] != 5, "roadmap of seed {} panics at iteration {} (code {})", seeds[r], sizes[4 * r], panic_code[r]);
        }
        (0..n)
            .map(|r| {
                let mut pto = PTO::new(self.fns);
                let s = [sizes[4 * r], sizes[4 * r + 1], sizes[4 * r + 2], sizes[4 * r + 3]];
                pto.copy_back_b200(r as i32, &s);
                (pto, if status[r] == 0 { Ok(()) } else { Err("final nodes are not reached for each world") })
            })
            .collect()
    }

    /// roadmap r of the ctx's last growth (`porrt_pto_fetch_roadmap`, sizes = iterations, nodes, directed edges, final nodes) into
    /// this planner's graph, kd-tree, reachability and n_it, bit for bit what `grow_graph` builds
    fn copy_back_b200(&mut self, r: i32, sizes: &[i64; 4]) {
        let ctx = self.fns.ctx;
        let mw = self.fns.mask_words();
        let (v, e, n_finals) = (sizes[1] as usize, sizes[2] as usize, sizes[3] as usize);
        let mut xy = vec![0f64; 2 * v];
        let mut node_vid = vec![0i32; v];
        let mut row_ptr = vec![0i64; v + 1];
        let (mut col, mut edge_vid) = (vec![0i32; e], vec![0i32; e]);
        let mut reach = vec![0u64; v * mw];
        let (mut fin_ids, mut fin_masks) = (vec![0i64; n_finals], vec![0u64; n_finals * mw]);
        ctx.check(unsafe {
            porrt_pto_fetch_roadmap(ctx.raw(), r, xy.as_mut_ptr(), node_vid.as_mut_ptr(), row_ptr.as_mut_ptr(), col.as_mut_ptr(),
                                    edge_vid.as_mut_ptr(), reach.as_mut_ptr(), fin_ids.as_mut_ptr(), fin_masks.as_mut_ptr())
        });
        let n_worlds = self.n_worlds;
        for k in 0..v {
            self.graph.add_node([xy[2 * k], xy[2 * k + 1]], node_vid[k] as usize);
            self.kdtree.add([xy[2 * k], xy[2 * k + 1]], k);
        }
        for u in 0..v {
            let (a, b) = (row_ptr[u] as usize, row_ptr[u + 1] as usize);
            let row: Vec<PTOEdge> = (a..b).map(|k| PTOEdge { id: col[k] as usize, validity_id: edge_vid[k] as usize }).collect();
            self.graph.nodes[u].parents = row.clone(); // parents(k) == children(k) as sequences (pto.rs:111-120)
            self.graph.nodes[u].children = row;
        }
        // Reachability (pto_reachability.rs) through its own API: the add_edge calls of pto.rs:111-120 replayed in insertion order --
        // the early part of row k (columns < k, kd order) is what node k added -- give the device's masks back bit for bit
        let validities = self.fns.world_validities();
        self.conservative_reachability.set_root(validities[node_vid[0] as usize].clone());
        for k in 1..v {
            self.conservative_reachability.add_node(validities[node_vid[k] as usize].clone());
            let early: Vec<&PTOEdge> = self.graph.nodes[k].children.iter().filter(|c| c.id < k).collect();
            for c in &early {
                self.conservative_reachability.add_edge(c.id, k, &validities[c.validity_id]);
            }
            for c in &early {
                self.conservative_reachability.add_edge(k, c.id, &validities[c.validity_id]);
            }
        }
        debug_assert!((0..v).all(|k| *self.conservative_reachability.reachability(k) == mask_from_words(&reach[k * mw..(k + 1) * mw], n_worlds)));
        for k in 0..n_finals {
            self.conservative_reachability.add_final_node(fin_ids[k] as usize, &mask_from_words(&fin_masks[k * mw..(k + 1) * mw], n_worlds));
        }
        self.n_it = sizes[0] as usize;
    }

    pub fn plan_belief_space_b200(&mut self, start_belief_state: &BeliefState) -> Policy<2> {
        assert_belief_state_validity(start_belief_state);
        let ctx = self.fns.ctx;
        let beliefs = self.fns.reachable_belief_states(start_belief_state);
        let b = beliefs.len();
        let n_worlds = self.n_worlds;
        let flat_beliefs: Vec<f64> = beliefs.iter().flatten().copied().collect();
        let (row_ptr, col, edge_vid, xy, node_vid) = export_csr(&self.graph);
        let v = self.graph.nodes.len();
        let states: Vec<[f64; 2]> = self.graph.nodes.iter().map(|n| n.state).collect();
        let visible = self.fns.visible_zones(&states); // observe()'s geometric test, once per node instead of once per (node, belief)
        let mw = self.fns.mask_words();
        let validities: Vec<u64> = self.fns.world_validities().iter().flat_map(|m| words_from_mask(m, mw)).collect();
        let n_validities = (validities.len() / mw) as i32;
        // final nodes with their finality masks (pto.rs:263-271)
        let (mut fin_ids, mut fin_masks): (Vec<i32>, Vec<u64>) = (Vec::new(), Vec::new());
        for (&final_id, validity) in self.conservative_reachability.final_nodes_with_validities() {
            fin_ids.push(final_id as i32);
            fin_masks.extend(words_from_mask(validity, mw));
        }
        // the V x B tables stay in ctx-owned pinned memory (porrt_belief_result): no second 8 * V * B byte copy
        ctx.check(unsafe {
            porrt_belief_vi(ctx.raw(), v as i64, row_ptr.as_ptr(), col.as_ptr(), edge_vid.as_ptr(), xy.as_ptr(), node_vid.as_ptr(),
                            validities.as_ptr(), n_validities, mw as i32, n_worlds as i32, flat_beliefs.as_ptr(), b as i32,
                            visible.as_ptr(), fin_ids.as_ptr(), fin_masks.as_ptr(), fin_ids.len() as i32, std::ptr::null_mut(),
                            std::ptr::null_mut(), std::ptr::null_mut(), std::ptr::null_mut())
        });
        let (mut dist_ptr, mut type_ptr): (*const f64, *const u8) = (std::ptr::null(), std::ptr::null());
        ctx.check(unsafe { porrt_belief_result(ctx.raw(), &mut dist_ptr, &mut type_ptr, std::ptr::null_mut(), std::ptr::null_mut()) });
        self.expected_costs_to_goals = unsafe { std::slice::from_raw_parts(dist_ptr, v * b) }.to_vec();
        // policy nodes in the reference's creation order
        let mut cap = 4096i64;
        let (mut n, mut cost) = (0i64, 0.0f64);
        let (mut node, mut belief, mut parent, mut leaf);
        loop {
            node = vec![0i32; cap as usize];
            belief = vec![0i32; cap as usize];
            parent = vec![0i32; cap as usize];
            leaf = vec![0u8; cap as usize];
            let rc = unsafe {
                porrt_extract_policy(ctx.raw(), node.as_mut_ptr(), belief.as_mut_ptr(), parent.as_mut_ptr(), leaf.as_mut_ptr(), cap, &mut n, &mut cost)
            };
            if rc == 4 {
                cap = n;
                continue;
            }
            ctx.check(rc);
            break;
        }
        let mut policy: Policy<2> = Policy { nodes: Vec::new(), leafs: Vec::new(), expected_costs: cost };
        for k in 0..n as usize {
            let original_id = node[k] as usize * b + belief[k] as usize; // the dense belief node id of pto.rs:197-199
            let id = policy.add_node(&states[node[k] as usize], &beliefs[belief[k] as usize], original_id, leaf[k] != 0);
            if parent[k] >= 0 {
                policy.add_edge(parent[k] as usize, id);
            }
        }
        policy
    }
}
