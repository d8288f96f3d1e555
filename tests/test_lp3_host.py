"""LP3 on the CPU: the constructed jam worlds reach what they claim (block_lp3's queue boundaries, no
distance ties, every LP3 branch), and the library's lp3 and lp3_stored, compiled for the host,
return the oracle's result and fail index bit for bit on every programme of those worlds and on
synthetic programmes at LP3's edges."""
import numpy as np
import pytest

import _emul_lp
import _lp3_worlds as W
from oracle.rvo2_oracle import solve_lp

SHAPES = [(16, 32), (16, 64), (16, 128), (16, 256), (24, 32), (24, 64), (24, 128), (24, 256), (32, 32), (32, 64),
          (32, 128), (32, 256), (40, 64), (40, 128), (40, 256), (100, 128), (100, 256), (256, 256)]


@pytest.mark.parametrize("N,tpb", SHAPES)
def test_assembled_blocks_hit_every_queue_boundary(N, tpb):
    """Per-block LP3 totals (the oracle's counts) equal the boundary targets, and together they take
    block_lp3 through all of its regimes: nobody, every solver storing its programme, stored and
    recomputing warps side by side, and nobody storing (fewer dead columns than a warp: only where
    the block's agents can leave that few).  Blocks are those of the tile kernel: block b holds envs
    [b * epb, (b + 1) * epb)."""
    for k in (5, 10):
        b = W.assemble(N, tpb, k)
        assert list(b["totals"]) == W.block_targets(N, tpb)
        assert b["pos"].shape[0] == len(b["targets"]) * b["epb"]
        regimes = set()
        for t in b["totals"]:
            ns = W.nstored(int(t), tpb)
            regimes.add("none" if t == 0 else "stored" if ns == t else "mixed" if ns > 0 else "recompute")
        assert {"none", "stored"} <= regimes, regimes
        cap = b["epb"] * N
        assert ("recompute" in regimes) == (W.nstored(cap, tpb) == 0), regimes
        if tpb >= 128:
            assert "mixed" in regimes
    print(N, tpb, W.block_targets(N, tpb), [W.nstored(t, tpb) for t in W.block_targets(N, tpb)])


def test_block_targets_cover_the_full_block_where_envs_fill_it():
    assert W.block_targets(16, 256)[-3:] == [224, 255, 256]
    assert W.block_targets(24, 256)[-2:] == [224, 240]  # 10 envs x 24 = 240 agents: 255 / 256 unreachable
    assert W.nstored(256, 256) == 0 and W.nstored(255, 256) == 0 and W.nstored(129, 256) == 96
    assert W.nstored(128, 256) == 128 and W.nstored(160, 256) == 96 and W.nstored(224, 256) == 32


@pytest.mark.parametrize("N,tpb", [(16, 256), (40, 128), (256, 256)])
def test_worlds_have_no_distance_ties(N, tpb):
    """No agent has two others within neighborDist at bit-equal squared distance, so every agent of
    these worlds is held to bit-exactness (no tie exemption)."""
    b = W.assemble(N, tpb, 10)
    for e in range(b["pos"].shape[0]):
        assert not W.has_tie(b["pos"][e], 5.0), e
    hb = W.hetero_batch(32, 256, 10)
    for e in range(hb["pos"].shape[0]):
        assert not W.has_tie(hb["pos"][e], 5.0), e


def _solve_all(progs, variant):
    bad = []
    lp3 = 0
    for j, (lines, n_obst, vmax, pref) in enumerate(progs):
        fo, ro = solve_lp(lines, n_obst, vmax, pref)
        f, r = _emul_lp.emul_solve(lines, len(lines), n_obst, vmax, pref, variant)
        lp3 += fo < len(lines)
        if f != fo or r.tobytes() != ro.tobytes():
            bad.append((j, fo, f, ro, r))
    return bad, lp3


@pytest.mark.parametrize("variant", [_emul_lp.LP3, _emul_lp.LP3_STORED])
def test_host_lp3_equals_oracle_on_the_world_library(variant):
    """Every agent's first-step programme of the assembled worlds: same fail index, same bits."""
    progs = W.library_programmes()
    _emul_lp.reset_counters()
    bad, lp3 = _solve_all(progs, variant)
    c = _emul_lp.counters()
    assert not bad, bad[:3]
    assert lp3 > 10000
    rounds = c[_emul_lp.LP3_ROUNDS] if variant == _emul_lp.LP3 else c[_emul_lp.LP3_STORED_ROUNDS]
    print(f"variant {variant}: {len(progs)} programmes, {lp3} LP3, {rounds} rounds, "
          f"{c[_emul_lp.LP3_INFEASIBLE]} infeasible, {c[_emul_lp.PARALLEL_SKIPPED]} parallel skipped, "
          f"{c[_emul_lp.ANTIPARALLEL]} antiparallel midpoints")
    assert rounds >= lp3
    for slot in (_emul_lp.LP3_INFEASIBLE, _emul_lp.PARALLEL_SKIPPED, _emul_lp.ANTIPARALLEL):
        assert c[slot] > 0, slot
    # each form counts only its own rounds
    assert c[_emul_lp.LP3_STORED_ROUNDS if variant == _emul_lp.LP3 else _emul_lp.LP3_ROUNDS] == 0


def test_both_lp3_forms_take_the_same_rounds():
    """lp3 and lp3_stored are one algorithm: the same number of rounds and of infeasible rounds."""
    progs = W.library_programmes(k_values=(10,))
    counts = []
    for variant in (_emul_lp.LP3, _emul_lp.LP3_STORED):
        _emul_lp.reset_counters()
        _solve_all(progs, variant)
        counts.append(_emul_lp.counters())
    a, b = counts
    assert a[_emul_lp.LP3_ROUNDS] == b[_emul_lp.LP3_STORED_ROUNDS] > 0
    assert a[_emul_lp.LP3_INFEASIBLE] == b[_emul_lp.LP3_INFEASIBLE]


@pytest.mark.parametrize("variant", [_emul_lp.LP3, _emul_lp.LP3_STORED])
def test_host_lp3_equals_oracle_on_synthetic_edges(variant):
    """det exactly 0, +-kEps and one ulp either side, duplicates, infeasible obstacle sets, n = 1..22,
    preferred velocities inside and outside the speed circle."""
    progs = W.synthetic_programmes()
    assert {len(p[0]) for p in progs} >= set(range(1, 23))
    _emul_lp.reset_counters()
    bad, lp3 = _solve_all(progs, variant)
    c = _emul_lp.counters()
    assert not bad, bad[:3]
    assert lp3 > 500
    for slot in (_emul_lp.LP3_INFEASIBLE, _emul_lp.PARALLEL_SKIPPED, _emul_lp.ANTIPARALLEL):
        assert c[slot] > 0, slot


def test_kEps_boundary_takes_the_parallel_branch_exactly_at_kEps():
    """One programme per side of the boundary: |det| = kEps is parallel (the projection is skipped or
    becomes a midpoint), one ulp above it is not -- counted by the host build, matched by the oracle."""
    up = np.nextafter(W.KEPS, np.float32(1))
    seen = {}
    for y, want_parallel in ((np.float32(0), True), (W.KEPS, True), (-W.KEPS, True), (up, False), (-up, False)):
        for s, slot in ((1, _emul_lp.PARALLEL_SKIPPED), (-1, _emul_lp.ANTIPARALLEL)):
            # line i: y >= 2 (outside the unit disc); line j before it with det(dir_i, dir_j) = y exactly
            lines = np.array([[0.0, -0.5, s * 1.0, y], [0.0, 2.0, 1.0, 0.0]], np.float32)
            _emul_lp.reset_counters()
            for variant in (_emul_lp.LP3, _emul_lp.LP3_STORED):
                fo, ro = solve_lp(lines, 0, 1.0, (0.0, 0.0))
                f, r = _emul_lp.emul_solve(lines, 2, 0, 1.0, (0.0, 0.0), variant)
                assert f == fo == 1 and r.tobytes() == ro.tobytes(), (y, s, variant)
            seen[(float(y), s)] = _emul_lp.counters()[slot]
            assert (seen[(float(y), s)] > 0) == want_parallel, (y, s)
