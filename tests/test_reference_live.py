"""Runs the UNMODIFIED reference shells and checks that the committed fixtures are what they
produce -- i.e. tests/golden/shell_*.npz are reproducible from the reference +
tests/golden/make_shell_golden.py.  The repository does not vendor the reference: these tests run
only where COLLISION_AVOIDANCE_REFERENCE names a checkout of it, and are skipped elsewhere."""
import contextlib
import io
import os
import sys

import numpy as np
import pytest

import _ref_stubs
from _golden import GOLDEN, load_alan, load_env

pytestmark = pytest.mark.skipif(not _ref_stubs.reference_available(), reason="needs COLLISION_AVOIDANCE_REFERENCE = a checkout of the reference project")


@pytest.fixture(scope="module")
def gen():
    from oracle import rvo2_oracle
    mods = _ref_stubs.load_reference(rvo2_oracle.PyRVOSimulator)
    sys.path.insert(0, GOLDEN)
    import make_shell_golden
    return make_shell_golden, mods


def _same(a, b):
    for k in b:
        assert np.array_equal(np.asarray(a[k]), b[k]), k


def test_alan_fixture_regenerates_from_the_reference(gen):
    g, (alan_mod, env_mod, train_mod) = gen
    name, n, act, seed, rec = g.ALAN_RUNS[1]
    _same(g.gen_alan_run(alan_mod, name, n, g.read_act(act), seed, rec, mode=1), load_alan("shell_alan_%s%d" % (name, n)))


def test_orca_fixture_regenerates_from_the_reference(gen):
    g, (alan_mod, env_mod, train_mod) = gen
    name, n, seed, rec = g.ORCA_RUNS[1]
    _same(g.gen_alan_run(alan_mod, name, n, None, seed, rec, mode=0), load_alan("shell_orca_%s%d" % (name, n)))


def test_env_fixture_regenerates_from_the_reference(gen):
    g, (alan_mod, env_mod, train_mod) = gen
    with contextlib.redirect_stdout(io.StringIO()):
        r = g.gen_env_run(env_mod, seed=303, n=2, steps_a=1000, steps_b=30, steps_orca=0, stop_on_done=True)
    _same(r, load_env("shell_env_small"))


def test_reference_registers_the_gym_id(gen):
    assert _ref_stubs.REGISTRY == {"collision_avoidance-v0": "collision_avoidance.envs:Collision_Avoidance_Env"}
