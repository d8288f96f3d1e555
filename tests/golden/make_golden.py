#!/usr/bin/env python
"""Generates the committed golden fixtures from the REFERENCE ITSELF (run with
COLLISION_AVOIDANCE_REFERENCE naming a checkout of it; the fixtures are committed, the reference
is not).

  laser_golden.npz   inputs + outputs of the reference's own utils.comp_laser /
                     utils.line_intersection (collision_avoidance/envs/utils.py:5-113)
  act_tables.json    the six trained ALAN action sets parsed from
                     collision_avoidance/ALAN/*_actions.act (Python-literal lists)
"""
import ast
import importlib.util
import json
import os
from math import cos, pi, sin

import numpy as np

REF = os.path.join(os.environ.get("COLLISION_AVOIDANCE_REFERENCE", ""), "collision_avoidance")
HERE = os.path.dirname(os.path.abspath(__file__))


def load_utils():
    spec = importlib.util.spec_from_file_location("ref_utils", os.path.join(REF, "envs", "utils.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def main():
    ref = load_utils()
    rng = np.random.default_rng(20261018)
    nd, r = 1.5, 0.5
    rays = [((0, 0), (nd * cos(i * 2 * pi / 16), -nd * sin(i * 2 * pi / 16))) for i in range(16)]
    octagon = []
    pts = [(r * cos(i * 2 * pi / 8), -r * sin(i * 2 * pi / 8)) for i in range(8)]
    for i in range(8):
        octagon.append((pts[i], pts[(i + 1) % 8]))
    cases = 200
    max_lines = 48
    seg = np.zeros((cases, max_lines, 4))
    vel = np.zeros((cases, max_lines, 2))
    nlines = np.zeros(cases, np.int64)
    orient = np.zeros((cases, 2))
    out = np.zeros((cases, 16, 4))
    for c in range(cases):
        lines = []
        for _ in range(int(rng.integers(0, 6))):  # neighbor octagons
            rel = rng.uniform(-1.6, 1.6, 2)
            v = tuple(rng.uniform(-1, 1, 2))
            for a, b in octagon:
                lines.append((((a[0] + rel[0], a[1] + rel[1]), (b[0] + rel[0], b[1] + rel[1])), v))
        for _ in range(int(rng.integers(0, 4))):  # wall segments
            a = rng.uniform(-2.5, 2.5, 2)
            b = a + rng.uniform(-3, 3, 2)
            lines.append(((tuple(a), tuple(b)), (0, 0)))
        lines = lines[:max_lines]
        ang = rng.uniform(-pi, pi)
        o = (cos(ang), sin(ang))
        orient[c] = o
        nlines[c] = len(lines)
        for k, ((a, b), v) in enumerate(lines):
            seg[c, k] = [a[0], a[1], b[0], b[1]]
            vel[c, k] = v
        if lines:
            res = ref.comp_laser(rays, lines, o)
        else:
            res = [((0, 0), (0, 0))] * 16
        for k, (hit, v) in enumerate(res):
            out[c, k] = [hit[0], hit[1], v[0], v[1]]
    # raw line_intersection cases
    li_in = rng.uniform(-2, 2, (500, 8))
    li_in[:, 0:2] = 0.0  # rays start at the origin like the laser
    li_d = np.zeros(500)
    li_p = np.zeros((500, 2))
    for k in range(500):
        d, pnt = ref.line_intersection(((li_in[k, 0], li_in[k, 1]), (li_in[k, 2], li_in[k, 3])),
                                       ((li_in[k, 4], li_in[k, 5]), (li_in[k, 6], li_in[k, 7])))
        li_d[k] = d
        li_p[k] = pnt
    np.savez_compressed(os.path.join(HERE, "laser_golden.npz"), seg=seg, vel=vel, nlines=nlines, orient=orient, out=out,
                        li_in=li_in, li_d=li_d, li_p=li_p)
    tables = {}
    for name in ("blocks", "circle", "congested", "crowd", "deadlock", "incoming"):
        with open(os.path.join(REF, "ALAN", f"{name}_actions.act")) as f:
            tables[name] = [list(map(float, t)) for t in ast.literal_eval(f.read().strip())]
    with open(os.path.join(HERE, "act_tables.json"), "w") as f:
        json.dump(tables, f, indent=1)
    print("wrote laser_golden.npz (", cases, "cases ) and act_tables.json", {k: len(v) for k, v in tables.items()})


if __name__ == "__main__":
    main()
