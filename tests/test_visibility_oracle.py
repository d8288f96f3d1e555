"""Known answers of the oracle's queryVisibility and roadmap (tests/host_emul/roadmap_oracle.cpp):
RVO2's line-of-sight recursion and Roadmap.cpp's buildRoadmap on hand-checked geometry."""
import numpy as np

from _roadmap_oracle import oracle_world

# counter-clockwise (RVO2's orientation for a solid obstacle): the inside is left of every edge
SQUARE = [(-1.0, -1.0), (1.0, -1.0), (1.0, 1.0), (-1.0, 1.0)]
# the same square moved up: its bottom edge y = 1 runs 1 unit beside the x axis
RAISED = [(-1.0, 1.0), (1.0, 1.0), (1.0, 3.0), (-1.0, 3.0)]


def test_empty_world_sees_everything():
    s = oracle_world([])
    for q1, q2, r in (((0, 0), (10, 3), 0.0), ((-5, 2), (5, -2), 100.0), ((1, 1), (1, 1), 1.0)):
        assert s.queryVisibility(q1, q2, r)


def test_before_process_obstacles_everything_is_visible():
    s = oracle_world([SQUARE], process=False)
    assert s.queryVisibility((-5, 0), (5, 0), 0.0)
    s.processObstacles()
    assert not s.queryVisibility((-5, 0), (5, 0), 0.0)


def test_wall_between_the_points_blocks():
    s = oracle_world([SQUARE])
    assert not s.queryVisibility((-5, 0), (5, 0), 0.0)
    assert not s.queryVisibility((5, 0.5), (-5, -0.5), 0.0)
    assert not s.queryVisibility((0, -5), (0, 5), 0.5)
    # a two-vertex obstacle is a wall that blocks from both sides
    w = oracle_world([[(0.0, -2.0), (0.0, 2.0)]])
    assert not w.queryVisibility((-1, 0), (1, 0), 0.0)
    assert not w.queryVisibility((1, 0), (-1, 0), 0.0)
    assert w.queryVisibility((-1, 3), (1, 3), 0.0)


def test_wall_beside_the_segment_blocks_when_radius_exceeds_the_clearance():
    s = oracle_world([RAISED])
    q1, q2 = (-5.0, 0.0), (5.0, 0.0)  # clearance 1 to the bottom edge
    one = np.float32(1.0)
    below = float(np.nextafter(one, np.float32(0)))
    above = float(np.nextafter(one, np.float32(2)))
    assert s.queryVisibility(q1, q2, 0.0)
    assert s.queryVisibility(q1, q2, 0.5)
    assert s.queryVisibility(q1, q2, below)
    # clearance exactly the radius: the edge's own test (>=) passes and the block is not searched
    assert s.queryVisibility(q1, q2, 1.0)
    # just above: the block is searched, and its side edges cross the segment within the radius
    assert not s.queryVisibility(q1, q2, above)
    assert not s.queryVisibility(q1, q2, 2.0)
    # a short segment whose line crosses no edge of the block is never blocked, whatever the radius:
    # RVO2 only blocks at edges whose line the segment crosses (or that come within the radius of it)
    assert s.queryVisibility((-0.5, 0.0), (0.5, 0.0), above)


def test_one_way_out_of_a_polygon():
    s = oracle_world([SQUARE])
    # from inside, the query leaves through the right edge: left-to-right is see-through
    assert s.queryVisibility((0, 0), (5, 0), 0.0)
    # coming in from outside crosses the edge: blocked
    assert not s.queryVisibility((5, 0), (0, 0), 0.0)


def test_segment_on_an_edge_supporting_line():
    s = oracle_world([SQUARE])
    # collinear with the bottom edge and off its end: the segment crosses no edge line
    assert s.queryVisibility((-5, -1), (-3, -1), 0.0)
    assert s.queryVisibility((-5, -1), (-3, -1), 0.5)
    # grazing the whole edge along its line touches the corners: blocked
    assert not s.queryVisibility((-5, -1), (5, -1), 0.0)


def test_degenerate_query_q1_equals_q2():
    s = oracle_world([SQUARE])
    # q1 == q2 gives a == b at every node: cases 1 and 2 only, and those never fail
    for p in ((5.0, 0.0), (0.0, 0.0), (1.0, 1.0), (1.5, 0.0)):
        for r in (0.0, 0.7, 10.0):
            assert s.queryVisibility(p, p, r)


def test_roadmap_edge_direction_and_unreachable_distance():
    s = oracle_world([SQUARE])
    inside, outside = (0.0, 0.0), (5.0, 0.0)
    # goal inside: the edge inside -> outside exists (inside sees out), so outside gets a distance
    adj, dist = s.roadmap_build([inside, outside], 1, 0.0)
    assert adj.tolist() == [[True, True], [False, True]]
    assert dist.tolist() == [[0.0, 5.0]]
    # goal outside: no edge leads from it to the inside vertex, which stays at 9e9f
    adj, dist = s.roadmap_build([outside, inside], 1, 0.0)
    assert adj.tolist() == [[True, False], [True, True]]
    assert dist[0, 0] == 0.0 and dist[0, 1] == np.float32(9e9)
