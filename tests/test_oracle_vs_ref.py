"""Pins the widened CPU restatement (oracle/nudge_oracle.cpp) to the UNMODIFIED reference, bit for bit, at every stage of the step
(SURVEY.md §8c): the oracle's stages, in the reference's layout, against digests of the reference's own stages recorded by
tests/golden/make_ref_traces.py.  CPU only; needs neither the reference nor oracle/_ref (tests/fuzz_oracle_vs_ref.py runs the same
comparison live where the reference is built)."""
import numpy as np
from nudge_b200 import scenes
from tests import golden_util as G
from tests.parity_util import ref_layout_stages, stage_digest


def _check_traces(name):
    """Runs the oracle through every case of `name` against the reference's trace; returns the sleeping pair count of every step."""
    from oracle import pyoracle
    g = G.load_ref_traces()
    sleeping = []
    for case, s, steps, cap, hook in G.ref_trace_cases(name):
        want = g[case]
        assert want.shape[0] == steps, case
        o = pyoracle.OracleSim(s, contact_capacity=cap)
        for i in range(steps):
            if hook:
                hook(i, o)
            got = [(stage, stage_digest(a)) for stage, a in ref_layout_stages(o, True)]
            sleeping.append(o.contacts.sleeping_count)
            if want.shape[1] == 1:      # one digest for the whole step (fuzz cases)
                assert stage_digest(np.array([d for _, d in got], np.uint64)) == want[i, 0], "%s (%s) step %d differs from the reference" % (case, s.name, i)
                continue
            assert len(got) == want.shape[1], "%s step %d: %d stages, the reference trace has %d" % (case, i, len(got), want.shape[1])
            for (stage, d), w in zip(got, want[i]):
                assert d == w, "%s step %d: %s differs from the reference" % (case, i, stage)
    return sleeping


def test_small_mixed_scene_every_stage():
    _check_traces("small_mixed")


def test_demo_scene_config0():
    """BASELINE config 0: 1024 boxes + 1024 spheres + ground, 8 iterations."""
    _check_traces("demo_config0")


def test_rotated_box_drop():
    _check_traces("rotated_box_drop")


def test_sleeping_islands_and_culled_cache():
    """Forces part of the scene asleep (idle counter 0xff) after 40 steps so that both island passes, sleeping pairs and the culled
    cache entries (nudge.cpp:3674-3700, 3973-4000, 4064-4101) are exercised."""
    sleeping = _check_traces("sleeping_islands")
    assert max(sleeping[40:]) > 0, "scenario never produced sleeping pairs"


def test_staged_calls_equal_fused_reference_step():
    """The seven calls made one by one (as the oracle and the GPU path make them) reproduce 20 steps of the reference's fused step loop."""
    from oracle import pyoracle
    g = G.load_ref_traces()
    s = scenes.demo_scene(64, 64, iterations=8, spread=2.0, height=10.0)
    o = pyoracle.OracleSim(s)
    for _ in range(20):
        o.step_staged()
    assert np.array_equal(o.transforms.view(np.uint8), g["fused_transforms"].view(np.uint8))
    assert np.array_equal(o.momentum.view(np.uint8), g["fused_momentum"].view(np.uint8))


def test_random_scenes_differential_fuzz_seeded():
    """A bounded, seeded run of tests/fuzz_oracle_vs_ref.py (random scenes, iterations, connections, sleep) against the reference's
    recorded steps: every stage of every step bit for bit."""
    _check_traces("fuzz")
