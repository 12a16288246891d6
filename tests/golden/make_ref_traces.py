"""Generates tests/golden/ref_traces.npz by running the UNMODIFIED reference (oracle/_ref, built by `make -C oracle ref`) through the
step sequences of tests/test_oracle_vs_ref.py (tests/golden_util.ref_trace_cases).  For every step of every case it stores one 8-byte
digest per stage (tests/parity_util.ref_layout_stages: contacts, tags, impulses, rows, momentum after every sweep, cache, transforms ...),
so the tests pin the widened oracle to the reference bit for bit without the reference.  For the 120 random scenes of the fuzz case one
digest per step, taken over its stage digests, keeps the file small (tests/fuzz_oracle_vs_ref.py finds the stage where the reference is
built).  It also stores the transforms and momentum after 20 fused reference steps (the reference's own step loop in one call), which the
oracle's seven staged calls must reproduce.
Run from the repo root where the reference is built:  python tests/golden/make_ref_traces.py"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np
from nudge_b200 import scenes as S
from oracle import pyref
from tests import golden_util as G
from tests.parity_util import ref_layout_stages, stage_digest


def trace(scene, steps, cap, hook, per_stage):
    r = pyref.RefSim(scene, contact_capacity=cap, arena_mb=1024)
    out, sleeping = [], 0
    for i in range(steps):
        if hook:
            hook(i, r)
        d = np.array([stage_digest(a) for _, a in ref_layout_stages(r, False)], np.uint64)
        out.append(d if per_stage else [stage_digest(d)])
        sleeping = max(sleeping, r.contacts.sleeping_count)
    return np.array(out, np.uint64), sleeping


def main():
    arr = {}
    for name in ("small_mixed", "demo_config0", "rotated_box_drop", "sleeping_islands", "fuzz"):
        for case, s, steps, cap, hook in G.ref_trace_cases(name):
            arr[case], sleeping = trace(s, steps, cap, hook, per_stage=name != "fuzz")
            if case == "sleeping_islands":
                assert sleeping > 0, "scenario never produced sleeping pairs"
    s = S.demo_scene(64, 64, iterations=8, spread=2.0, height=10.0)
    a = pyref.RefSim(s); b = pyref.RefSim(s)
    for _ in range(20):
        a.step(); b.step_staged()
    assert a.transforms.tobytes() == b.transforms.tobytes() and a.momentum.tobytes() == b.momentum.tobytes()
    arr["fused_transforms"], arr["fused_momentum"] = a.transforms, a.momentum
    here = os.path.dirname(os.path.abspath(__file__))
    np.savez_compressed(os.path.join(here, "ref_traces.npz"), **arr)
    print("cases", len(arr) - 2, "digests", sum(v.size for k, v in arr.items() if not k.startswith("fused")))


if __name__ == "__main__":
    main()
