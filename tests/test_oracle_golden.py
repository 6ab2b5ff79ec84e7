"""Pins the CPU oracle against the reference's own MAP-FREE golden tests (SURVEY.md 8(c)).

Each test names the reference test it transcribes (file:line under /root/reference/src).
"""
import math

import numpy as np
import pytest

from oracle import pyoracle as O

INF = float("inf")


# ------------------------------------------------------------------ nearest_neighbor.rs:142-311
NODES = [[3.0, 6.0], [17.0, 15.0], [13.0, 15.0], [6.0, 12.0], [9.0, 1.0], [2.0, 7.0], [10.0, 19.0]]
CENTERS = [[17.0, 15.0], [9.1, 1.0], [2.0, 8.0], [15.0, 13.0], [3.0, 5.0], [13.0, 7.0]]


def create_tree():
    tree = O.KdTree(NODES[0])
    for i, n in enumerate(NODES[1:]):
        tree.add(n, i + 1)
    return tree


def test_kdtree_creation():  # nearest_neighbor.rs:170-177
    ids, left, right, _ = O.KdTree([3.0, 6.0]).export()
    assert list(ids) == [0] and left[0] == -1 and right[0] == -1


def test_add_second_level():  # :179-195
    t = O.KdTree([3.0, 6.0])
    t.add([2.0, 7.0], 1)
    ids, left, right, xy = t.export()
    assert right[0] == -1 and ids[left[0]] == 1 and list(xy[left[0]]) == [2.0, 7.0]
    t = O.KdTree([3.0, 6.0])
    t.add([17.0, 15.0], 1)
    ids, left, right, xy = t.export()
    assert left[0] == -1 and ids[right[0]] == 1 and list(xy[right[0]]) == [17.0, 15.0]


def test_full_tree():  # :197-234
    ids, left, right, xy = create_tree().export()

    def chk(slot, id, state):
        assert ids[slot] == id and list(xy[slot]) == state

    chk(left[0], 5, [2.0, 7.0])
    chk(right[0], 1, [17.0, 15.0])
    chk(left[right[0]], 3, [6.0, 12.0])
    chk(right[right[0]], 2, [13.0, 15.0])
    chk(right[left[right[0]]], 4, [9.0, 1.0])
    chk(left[right[right[0]]], 6, [10.0, 19.0])


def test_nearest_neighbor_vs_brute_force():  # :237-265
    tree = create_tree()
    for c in CENTERS:
        d = sorted(((math.sqrt((n[0] - c[0]) ** 2 + (n[1] - c[1]) ** 2), i) for i, n in enumerate(NODES)))
        assert tree.nearest_neighbor(c) == d[0][1]
        for radius in range(1, 10):
            expect = sorted(i for dist, i in d if dist <= radius)
            assert sorted(tree.nearest_neighbors(c, float(radius))) == expect


def test_nearest_neighbor_with_filter():  # :267-311
    tree = create_tree()
    seq = [(0, []), (5, [0]), (3, [0, 5]), (4, [0, 5, 3]), (2, [0, 5, 3, 4]), (6, [0, 5, 3, 4, 2]), (1, [0, 5, 3, 4, 2, 6])]
    for expect, excl in seq:
        assert tree.nearest_neighbor([3.1, 6.0], excl) == expect
    seq = [(2, []), (1, [2]), (6, [2, 1]), (3, [2, 1, 6])]
    for expect, excl in seq:
        assert tree.nearest_neighbor([13.0, 15.1], excl) == expect


def test_radius_order_is_kd_preorder():
    # result order = node, left, right (nearest_neighbor.rs:101-117)
    tree = create_tree()
    assert list(tree.nearest_neighbors([9.0, 10.0], 100.0)) == [0, 5, 1, 3, 4, 2, 6]


# ------------------------------------------------------------------ pto_graph.rs:434-700
def minimal_graph():
    g = O.PTOGraph([[1]])
    g.add_node([0.0, 0.0], 0)
    g.add_node([1.0, 0.0], 0)
    g.add_edge(0, 1, 0)
    return g


def grid_graph():
    g = O.PTOGraph([[1]])
    for y in range(3):
        for x in range(3):
            g.add_node([float(x), float(y)], 0)
    for a, b in [(0, 1), (1, 2), (0, 3), (1, 4), (2, 5), (3, 4), (4, 5), (3, 6), (4, 7), (5, 8), (6, 7), (7, 8)]:
        g.add_bi_edge(a, b, 0)
    return g


def oriented_grid_graph():
    g = O.PTOGraph([[1]])
    for s in ([0.0, 0.0], [1.0, 0.0], [0.0, 1.0], [1.0, 1.0]):
        g.add_node(s, 0)
    for a, b in [(0, 1), (0, 2), (1, 3), (3, 2)]:
        g.add_edge(a, b, 0)
    return g


def diamond_graph_2_worlds():
    g = O.PTOGraph([[1, 0], [0, 1], [1, 1]])
    g.add_node([0.0, 0.0], 2)
    g.add_node([1.0, 1.0], 1)
    g.add_node([1.0, -1.0], 0)
    g.add_node([2.0, 0.0], 2)
    g.add_bi_edge(0, 1, 0)
    g.add_bi_edge(0, 2, 1)
    g.add_bi_edge(1, 3, 0)
    g.add_bi_edge(2, 3, 1)
    return g


def test_dijkstra_on_minimal_graph():  # :625-634
    assert list(minimal_graph().dijkstra([1])) == [1.0, 0.0]


def test_dijkstra_on_grid_graph_single_goal():  # :636-645
    assert list(grid_graph().dijkstra([8])) == [4.0, 3.0, 2.0, 3.0, 2.0, 1.0, 2.0, 1.0, 0.0]


def test_dijkstra_on_grid_graph_two_goals():  # :647-656
    assert list(grid_graph().dijkstra([7, 5])) == [3.0, 2.0, 1.0, 2.0, 1.0, 0.0, 1.0, 0.0, 1.0]


def test_dijkstra_without_final_node():  # :658-667
    assert list(grid_graph().dijkstra([])) == [INF] * 9


def test_dijkstra_on_oriented_grid():  # :669-678
    assert list(oriented_grid_graph().dijkstra([3])) == [2.0, 1.0, INF, 0.0]


def test_dijkstra_world_views():  # the dijkstra calls of :591-606
    g = diamond_graph_2_worlds()
    s2 = math.sqrt(2.0)
    # world 0: node 1 (validity [0,1]) is invalid, node 2 (validity [1,0]) valid
    assert list(g.dijkstra([3], world=0)) == [s2 + s2, INF, s2, 0.0]
    assert list(g.dijkstra([3], world=1)) == [s2 + s2, s2, INF, 0.0]


def test_world_transitions():  # :680-700
    wv = [[1, 0], [0, 1], [1, 1]]
    assert O.default_transition_validator(wv, 0, 0) == 0
    assert O.default_transition_validator(wv, 0, 1) == O.NONE
    assert O.default_transition_validator(wv, 2, 2) == 2


# ------------------------------------------------------------------ belief_graph.rs:276-577
A, OBS = O.ACTION, O.OBSERVATION


def create_graph_1(bs):
    g = O.BeliefGraph(bs)
    spec = [([0.0, 1.0], 0, A), ([-1.0, 2.0], 0, A), ([1.0, 2.0], 0, A), ([0.0, 4.0], 0, A), ([0.0, 0.0], 0, OBS),
            ([0.0, 0.0], 1, A), ([0.0, 1.0], 1, A), ([-1.0, 2.0], 1, A), ([1.0, 2.0], 1, A), ([-1.0, 3.0], 1, A), ([0.0, 4.0], 1, A),
            ([0.0, 0.0], 2, A), ([0.0, 1.0], 2, A), ([-1.0, 2.0], 2, A), ([1.0, 2.0], 2, A), ([10.0, 3.0], 2, A), ([0.0, 4.0], 2, A)]
    for s, b, t in spec:
        g.add_node(s, b, t)

    def bi(a, b):
        g.add_edge(a, b)
        g.add_edge(b, a)

    bi(0, 1); bi(0, 2); g.add_edge(0, 4)
    g.add_edge(4, 5); bi(5, 6); bi(6, 7); bi(6, 8); bi(7, 9); bi(9, 10)
    g.add_edge(4, 11); bi(11, 12); bi(12, 13); bi(12, 14); bi(14, 15); bi(15, 16)
    return g


def create_graph_2(bs):
    # NB: the reference passes belief_states[1] as the *state vector* of nodes 18..27 but belief_id 2
    # (belief_graph.rs:452-461); only belief_id matters here because BeliefGraph::new gets an empty
    # reachable list in the reference test, while ours resolves belief states through belief_id.
    # To reproduce the reference's arithmetic (transition_probability on the node's stored belief_state)
    # the third belief row used for those nodes must equal belief_states[1].
    g = O.BeliefGraph([bs[0], bs[1], bs[1]])
    st0 = [[0.0, 0.0], [0.0, 1.0], [1.0, 0.0], [2.0, 0.0], [2.0, 1.0], [2.0, 2.0], [2.0, 3.0], [1.0, 3.0], [0.0, 3.0]]
    for k, s in enumerate(st0):
        g.add_node(s, 0, OBS if k == 1 else A)
    for s in st0:
        g.add_node(s, 1, A)
    st2 = [[0.0, 0.0], [0.0, 1.0], [0.0, 2.0], [1.0, 0.0], [2.0, 0.0], [2.0, 1.0], [2.0, 2.0], [2.0, 3.0], [1.0, 3.0], [0.0, 3.0]]
    for s in st2:
        g.add_node(s, 2, A)

    def bi(a, b):
        g.add_edge(a, b)
        g.add_edge(b, a)

    g.add_edge(0, 1); bi(0, 2); bi(2, 3); bi(3, 4); bi(4, 5); bi(5, 6); bi(6, 7); bi(7, 8)
    g.add_edge(1, 10); bi(10, 9); bi(9, 11); bi(11, 12); bi(12, 13); bi(13, 14); bi(14, 15); bi(15, 16); bi(16, 17)
    g.add_edge(1, 19); bi(19, 20); bi(20, 27); bi(19, 18); bi(18, 21); bi(21, 22); bi(22, 23); bi(23, 24); bi(24, 25)
    g.add_edge(26, 25); g.add_edge(25, 26); g.add_edge(27, 26); g.add_edge(26, 27)
    return g


def test_conditional_dijkstra_and_extract_policy_on_graph_1():  # :500-544
    bs = [[0.4, 0.6], [1.0, 0.0], [0.0, 1.0]]
    g = create_graph_1(bs)
    d = g.conditional_dijkstra([3, 10, 16])
    assert d[0] < d[1] and d[0] < d[2] and d[4] < d[0]
    assert d[6] < d[5] and d[6] < d[8] and d[7] < d[6] and d[9] < d[7] and d[10] < d[9]
    assert d[12] < d[11] and d[12] < d[13] and d[14] < d[12] and d[15] < d[14] and d[16] < d[15]
    assert d[4] == bs[0][0] * d[5] + bs[0][1] * d[11]  # :528
    pol = g.extract_policy(d)
    assert len(pol.leafs) == 2
    assert tuple(pol.xy[pol.leafs[0]]) == (0.0, 4.0) and tuple(pol.xy[pol.leafs[1]]) == (0.0, 4.0)
    assert pol.belief_id[pol.leafs[0]] == 2 and pol.belief_id[pol.leafs[1]] == 1  # "second belief first"
    assert pol.path_to_leaf(0) == [(0.0, 1.0), (0.0, 0.0), (0.0, 0.0), (0.0, 1.0), (1.0, 2.0), (10.0, 3.0), (0.0, 4.0)]
    assert pol.path_to_leaf(1) == [(0.0, 1.0), (0.0, 0.0), (0.0, 0.0), (0.0, 1.0), (-1.0, 2.0), (-1.0, 3.0), (0.0, 4.0)]


def test_conditional_dijkstra_and_extract_policy_on_graph_2():  # :546-567
    bs = [[0.4, 0.6], [1.0, 0.0], [0.0, 1.0]]
    g = create_graph_2(bs)
    d = g.conditional_dijkstra([8, 17, 27])
    mi, md = 0, 0.0
    for i, v in enumerate(d):
        if v > md:
            mi, md = i, v
    assert mi == 10 and md == 8.0
    pol = g.extract_policy(d)
    assert len(pol.leafs) == 2
    assert tuple(pol.xy[pol.leafs[0]]) == (0.0, 3.0) and tuple(pol.xy[pol.leafs[1]]) == (0.0, 3.0)


def test_belief_state_hashing():  # :569-577
    h = lambda b: O.lib().orc_belief_hash(O.P(O.f64a(b)), len(b))
    assert h([2.0 / 3.0, 1.0 / 3.0]) != h([1.0 / 3.0, 2.0 / 3.0])
    assert len({h([0.5, 0.5]), h([1.0, 0.0]), h([0.0, 1.0])}) == 3
    assert h([0.5, 0.5]) == 2 * 500 + 11 * 500  # (10^0+1)*500 + (10^1+1)*500, common.rs:354


# ------------------------------------------------------------------ pto_reachability.rs:109-230
def test_reachability():
    r = O.Reachability()
    r.set_root([1, 1]); r.add_node([1, 0]); r.add_node([1, 0]); r.add_node([0, 1])
    r.add_edge(0, 1, [1, 0]); r.add_edge(1, 2, [1, 0]); r.add_edge(1, 3, [0, 1])
    assert [list(r.reachability(i)) for i in range(4)] == [[1, 1], [1, 0], [1, 0], [0, 0]]


def test_reachability_diamond_shape():
    r = O.Reachability()
    r.set_root([1, 1]); r.add_node([1, 0]); r.add_node([0, 1]); r.add_node([1, 1])
    r.add_edge(0, 1, [1, 0]); r.add_edge(0, 2, [0, 1]); r.add_edge(1, 3, [1, 1]); r.add_edge(2, 3, [1, 1])
    assert [list(r.reachability(i)) for i in range(4)] == [[1, 1], [1, 0], [0, 1], [1, 1]]


def test_final_nodes_completness():
    r = O.Reachability()
    r.set_root([1, 1]); r.add_node([1, 1]); r.add_node([1, 0]); r.add_node([0, 1])
    r.add_edge(0, 1, [1, 1]); r.add_edge(1, 2, [1, 0]); r.add_edge(1, 3, [0, 1])
    assert not r.is_final_set_complete()
    r.add_final_node(2, [1, 1])
    assert not r.is_final_set_complete()
    r.add_final_node(3, [1, 1])
    assert r.is_final_set_complete()
    assert r.get_final_nodes_for_world(0) == [2] and r.get_final_nodes_for_world(1) == [3]


def test_final_nodes_completness_2_goals_2_worlds():
    r = O.Reachability()
    r.set_root([1, 1]); r.add_node([1, 1]); r.add_node([1, 1]); r.add_node([1, 1])
    r.add_edge(0, 1, [1, 1]); r.add_edge(1, 2, [1, 1]); r.add_edge(1, 3, [1, 1])
    r.add_final_node(2, [1, 0])
    assert not r.is_final_set_complete()
    r.add_final_node(3, [0, 1])
    assert r.is_final_set_complete()
    assert r.get_final_nodes_for_world(0) == [2] and r.get_final_nodes_for_world(1) == [3]
    ids, fin = r.finals()
    assert list(ids) == [2, 3] and fin.tolist() == [[1, 0], [0, 1]]


# ------------------------------------------------------------------ common.rs:401-523
def test_goal():
    g = O.SquareGoal([([0.1, 0.1], [1, 0]), ([0.9, 0.9], [0, 1])], 0.1)
    assert list(g.goal([0.11, 0.11])) == [1, 0]
    assert g.goal([0.5, 0.5]) is None
    assert list(g.goal([0.91, 0.91])) == [0, 1]
    assert list(g.goal_example(0)) == [0.1, 0.1] and list(g.goal_example(1)) == [0.9, 0.9]


def test_transitions():
    tp = lambda p, c: O.lib().orc_transition_probability(O.P(O.f64a(p)), O.P(O.f64a(c)), len(p))
    assert tp([1.0, 0.0], [1.0, 0.0]) == 1.0
    assert tp([0.0, 1.0], [1.0, 0.0]) == 0.0
    assert tp([0.4, 0.6], [0.4, 0.6]) == 1.0
    assert tp([0.4, 0.6], [1.0, 0.0]) == 0.4
    assert tp([0.5, 0.0, 0.5, 0.0], [0.0, 0.5, 0.0, 0.5]) == 0.0


def test_norms_and_steer():
    n1 = O.lib().orc_norm1(O.P(O.f64a([0.0, 0.0])), O.P(O.f64a([3.0, -4.0])))
    n2 = O.lib().orc_norm2(O.P(O.f64a([0.0, 0.0])), O.P(O.f64a([3.0, -4.0])))
    assert n1 == 7.0 and n2 == 5.0
    to = O.f64a([1.0, 1.0])
    O.lib().orc_steer(O.P(O.f64a([0.0, 0.0])), O.P(to), 0.5)  # norm1 step = 2 -> lambda = 0.25
    assert list(to) == [0.25, 0.25]


def _reference_policy(beliefs0, last):
    """the policy of common.rs:425-489: 0 -> 1 -> {2, 3}, 2 -> 4, 3 -> 5 (nodes 1, 2, 3 share a state: the observation)"""
    xy = np.array([[0.0, 0.0], [0.0, 1.0], [0.0, 1.0], [0.0, 1.0], [-1.0, 2.0], last])
    beliefs = np.array([beliefs0, [1.0, 0.0], [0.0, 1.0]])
    belief_id = np.array([0, 0, 1, 2, 1, 2], np.int64)
    parent = np.array([-1, 0, 1, 1, 2, 3], np.int64)
    return xy, beliefs, belief_id, parent


def test_policy_decomposition():  # common.rs:425-457
    xy, beliefs, belief_id, parent = _reference_policy([0.5, 0.5], [1.0, 2.0])
    assert O.lib().orc_policy_decompose_count(O.P(parent), len(parent)) == 3
    import po_rrt_b200 as P                                   # the product's host-side row (no device needed)
    pieces, skeleton = P.policy_decompose(parent)
    assert len(pieces) == 3
    assert [p.tolist() for p in pieces] == [[0, 1], [2, 4], [3, 5]] and skeleton == [[1, 2], [], []]


def test_policy_expected_cost_computation():  # common.rs:459-489
    xy, beliefs, belief_id, parent = _reference_policy([0.4, 0.6], [2.0, 3.0])
    want = 1.0 + 0.4 * 2.0 ** 0.5 + 0.6 * 2.0 * 2.0 ** 0.5    # assert_eq!(policy.expected_costs, 1.0 + 0.4 * sqrt 2 + 0.6 * 2.0 * sqrt 2)
    got = O.lib().orc_policy_expected_cost(O.P(np.ascontiguousarray(xy)), O.P(belief_id), O.P(parent), len(parent), O.P(np.ascontiguousarray(beliefs)), 3, 2)
    assert got == want
    import po_rrt_b200 as P
    assert P.policy_expected_cost(xy, belief_id, parent, beliefs) == want


def test_wm_contains():  # common.rs:413-423 (contains() is used by nobody on the hot path; restated here only)
    contains = lambda a, b: all(x or not y for x, y in zip(a, b))
    assert contains([1, 1], [1, 1]) and contains([1, 1], [1, 0]) and contains([1, 1], [0, 1]) and contains([1, 1], [0, 0])
    assert contains([1, 0], [1, 0]) and not contains([1, 0], [0, 1]) and not contains([0, 0], [0, 1])


def test_heuristic_radius():  # common.rs:357-369 (test only prints; we pin the formula against libm)
    for n in (2, 10, 100, 1000, 10000, 1000000):
        s = 2.0 * (math.log(n) / n) ** 0.5
        assert O.lib().orc_heuristic_radius(n, 0.1, 2.0, 2) == min(s, 0.1) or abs(O.lib().orc_heuristic_radius(n, 0.1, 2.0, 2) - min(s, 0.1)) < 1e-15
    assert O.lib().orc_heuristic_radius(1, 0.1, 2.0, 2) == 0.0


# ------------------------------------------------------------------ third-party restatements
def test_pcg64_known_answer_vector():
    # official pcg64 (XSL-RR 128/64) demo vector for seed (42, 54)
    r = O.Pcg64.new(42, 54)
    assert [r.next_u64() for _ in range(3)] == [0x86b1da1d72062b68, 0x1304aa46c9853d39, 0xa3670e9e0dd50358]


def test_sampler_ranges():  # sample_space.rs:62-115 (range checks only)
    r = O.Pcg64(0)
    s = r.sample_states([-1.0, -0.5], [1.0, 0.5], 2000)
    assert (s[:, 0] >= -1.0).all() and (s[:, 0] < 1.0).all() and (s[:, 1] >= -0.5).all() and (s[:, 1] < 0.5).all()
    d = O.Pcg64(0)
    v = [d.gen_range_usize(3) for _ in range(500)]
    assert set(v) == {0, 1, 2}
    # two generators seeded alike agree (ContinuousSampler / DiscreteSampler both use seed 0)
    a, b = O.Pcg64(0), O.Pcg64(0)
    assert [a.next_u64() for _ in range(5)] == [b.next_u64() for _ in range(5)]


def test_bresenham_doc_example_and_closed_form():
    # line_drawing 0.8 doc example
    assert O.bresenham((0, 0), (5, 6)).tolist() == [[0, 0], [0, 1], [1, 2], [2, 3], [3, 4], [4, 5], [5, 6]]
    assert O.bresenham((0, 0), (5, 2)).tolist() == [[0, 0], [1, 0], [2, 0], [3, 1], [4, 1], [5, 2]]
    assert O.bresenham((3, 3), (3, 3)).tolist() == [[3, 3]]
    # closed form used by the CUDA kernels (SURVEY 8(a) A5): pixel k = from_octant(x0+k, y0+floor(k*dy/dx))
    frm = {0: lambda x, y: (x, y), 1: lambda x, y: (y, x), 2: lambda x, y: (-y, x), 3: lambda x, y: (-x, y),
           4: lambda x, y: (-x, -y), 5: lambda x, y: (-y, -x), 6: lambda x, y: (y, -x), 7: lambda x, y: (x, -y)}
    to = {0: lambda x, y: (x, y), 1: lambda x, y: (y, x), 2: lambda x, y: (y, -x), 3: lambda x, y: (-x, y),
          4: lambda x, y: (-x, -y), 5: lambda x, y: (-y, -x), 6: lambda x, y: (-y, x), 7: lambda x, y: (x, -y)}
    rng = np.random.default_rng(1)
    pts = rng.integers(-40, 40, size=(400, 4))
    for ax, ay, bx, by in pts.tolist() + [[0, 0, 7, 7], [0, 0, -7, 7], [5, 5, 5, -9], [2, 1, -8, 1]]:
        dx, dy, o = bx - ax, by - ay, 0
        if dy < 0:
            dx, dy, o = -dx, -dy, o + 4
        if dx < 0:
            dx, dy, o = dy, -dx, o + 2
        if dx < dy:
            o += 1
        sx, sy = to[o](ax, ay)
        ex, ey = to[o](bx, by)
        ddx, ddy = ex - sx, ey - sy
        closed = [list(frm[o](sx + k, sy + (k * ddy // ddx if ddx else 0))) for k in range(ddx + 1)]
        assert O.bresenham((ax, ay), (bx, by)).tolist() == closed
        assert len(closed) == max(abs(bx - ax), abs(by - ay)) + 1


def test_fixed_point_minor_offset_is_exact():
    """edge3.cu: floor(k*dy/dx) == hi32(k*S + 2^16) for every 0 <= dy <= dx < 2^15 and 0 <= k <= dx (DESIGN.md 3.1),
    both for the exact S = min(floor(dy*2^32/dx), 2^32-1) and for the S the kernels compute on the FP64 pipe,
    trunc_sat(dy * 2^32 * rn(1/dx)) -- replayed here in IEEE double arithmetic (numpy division and multiplication are correctly
    rounded like __drcp_rn / __dmul_rn).  Exhaustive for dx <= 160, all dy / sampled k for large dx."""
    B = np.uint64(65536)
    for dx in list(range(1, 161)) + [255, 256, 257, 4095, 4096, 8191, 16383, 32767]:
        dy = np.arange(0, dx + 1, dtype=np.uint64)
        if dx > 160:
            dy = np.unique(np.concatenate([dy[:40], dy[-40:], dy[::max(1, dx // 97)]]))
        k = np.arange(0, dx + 1, dtype=np.uint64)
        want = (k[None, :] * dy[:, None]) // np.uint64(dx)
        S_exact = np.minimum((dy << np.uint64(32)) // np.uint64(dx), np.uint64(0xFFFFFFFF))
        S_fp = np.minimum(np.floor((dy.astype(np.float64) * 4294967296.0) * (1.0 / np.float64(dx))), 4294967295.0).astype(np.uint64)
        assert (np.abs(S_fp.astype(np.int64) - S_exact.astype(np.int64)) <= 1).all()
        for S in (S_exact, S_fp):
            got = (k[None, :] * S[:, None] + B) >> np.uint64(32)
            assert np.array_equal(got, want), dx
