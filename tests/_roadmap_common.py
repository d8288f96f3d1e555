"""Worlds, query endpoints and roadmaps shared by the roadmap tests (CPU and GPU)."""
import numpy as np

from collision_avoidance_b200 import scenarios

RADII = np.array([0.0, 0.1, 0.5, 2.0], np.float32)


def random_polygons(seed, n=6):
    """Star-shaped random polygons (some concave), counter-clockwise, inside an enclosing wall."""
    rng = np.random.default_rng(seed)
    polys = [[(-30.0, -30.0), (-30.0, 30.0), (30.0, 30.0), (30.0, -30.0)]]
    for _ in range(n):
        c = rng.uniform(-20, 20, 2)
        k = int(rng.integers(3, 8))
        ang = np.sort(rng.uniform(0, 2 * np.pi, k))
        rad = rng.uniform(1.0, 5.0, k)
        polys.append([(float(c[0] + r * np.cos(a)), float(c[1] + r * np.sin(a))) for a, r in zip(ang, rad)])
    return polys


def worlds():
    rb, _, _ = scenarios.roadmap_blocks(1)
    return {
        "blocks": scenarios.blocks(1, 8).obstacles[0],
        "deadlock": scenarios.deadlock(1, 10).obstacles,
        "congested": scenarios.congested(1, 12).obstacles,
        "default_env": scenarios.default_env(1).obstacles,
        "roadmap_blocks": rb.obstacles,
        "random_a": random_polygons(1),
        "random_b": random_polygons(2, n=12),
    }


def query_points(polys, n, rng):
    """Endpoints near vertices, on edge lines (inside and beyond the edges) and anywhere in the box."""
    v = np.concatenate([np.asarray(p, np.float32) for p in polys])
    nxt = np.concatenate([np.roll(np.arange(len(p)), -1) + off for p, off in
                          zip(polys, np.cumsum([0] + [len(p) for p in polys[:-1]]))])
    lo, hi = v.min(0), v.max(0)
    kind = rng.integers(0, 4, n)
    i = rng.integers(0, v.shape[0], n)
    scale = rng.choice(np.float32([0.0, 1e-3, 0.1, 1.0]), n)
    near = v[i] + scale[:, None] * rng.standard_normal((n, 2)).astype(np.float32)
    t = rng.uniform(-0.5, 1.5, n).astype(np.float32)[:, None]
    on_line = v[i] + t * (v[nxt[i]] - v[i])
    anywhere = rng.uniform(lo, hi, (n, 2)).astype(np.float32)
    vertex = v[i]
    out = np.where((kind == 0)[:, None], near, np.where((kind == 1)[:, None], on_line,
                                                          np.where((kind == 2)[:, None], anywhere, vertex)))
    return np.ascontiguousarray(out, np.float32)


def random_roadmap(polys, R, rng):
    v = np.concatenate([np.asarray(p, np.float32) for p in polys])
    lo, hi = v.min(0), v.max(0)
    pts = rng.uniform(lo, hi, (R, 2)).astype(np.float32)
    # a few vertices repeated and a few on obstacle corners
    if R > 4:
        pts[-1] = pts[0]
        pts[-2] = v[rng.integers(0, v.shape[0])]
    return pts
