#!/usr/bin/env python
"""Differential fuzz of the widened CPU oracle (oracle/nudge_oracle.cpp) against the UNMODIFIED reference compiled in place (oracle/_ref):
random box / sphere / mixed scenes, 1-20 solver iterations, random body connections, parts of the scene put to sleep on the way;
every stage of every step compared bit for bit (tests/parity_util.compare_ref_oracle_step).  CPU only, needs oracle/_ref.

    python tests/fuzz_oracle_vs_ref.py [seconds] [seed]        (round 2: 1500 s, seed 2026 -> 30,615 scenes, 0 mismatches)

Dense start states are avoided on purpose: the reference does not check its capacities (SURVEY.md section 0.8) and overruns the caller's
buffers when a scene produces more contacts than they hold."""
import os, sys, time
import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from nudge_b200 import scenes
from tests.parity_util import Report, compare_ref_oracle_step


def random_scene(rng):
    nb, ns = int(rng.integers(0, 400)), int(rng.integers(0, 400))
    if nb + ns == 0:
        nb = 8
    it = int(rng.choice([1, 4, 8, 20])); seed = int(rng.integers(0, 1 << 30))
    kind = int(rng.integers(0, 3))
    if kind == 0:
        s = scenes.demo_scene(nb, ns, iterations=it, spread=float(rng.uniform(3, 8)), height=float(rng.uniform(10, 60)), seed=seed)
    elif kind == 1:
        s = scenes.box_drop(max(nb, 8), iterations=it, seed=seed)
    else:
        s = scenes.mixed_stack(max(nb + ns, 16), iterations=it, seed=seed)
    if rng.random() < 0.3 and s.n_bodies > 4:
        k = int(rng.integers(1, 6))
        s.connections = np.zeros(k, scenes.PAIR32); s.connections["a"] = rng.integers(1, s.n_bodies, k); s.connections["b"] = rng.integers(1, s.n_bodies, k)
    return s


def contact_capacity(s):
    return 256 * s.n_bodies + 4096


def maybe_sleep(rng, sims):
    """Before a step: now and then put a random half of the scene to sleep in every sim of `sims`."""
    if rng.random() < 0.05:
        m = rng.random(sims[0].scene.n_bodies) < 0.5
        for x in sims:
            x.idle[m] = 0xff
            x.momentum["velocity"][m] = 0; x.momentum["angular_velocity"][m] = 0


def run_scene(s, rng, steps):
    """Returns None, or a description of the first difference."""
    from oracle import pyref, pyoracle
    r = pyref.RefSim(s, contact_capacity=contact_capacity(s), arena_mb=1024); o = pyoracle.OracleSim(s, contact_capacity=r.cap)
    for i in range(steps):
        maybe_sleep(rng, (r, o))
        rep = Report("%s step %d" % (s.name, i))
        if not compare_ref_oracle_step(r, o, rep):
            return str(rep)
    return None


def main():
    seconds = float(sys.argv[1]) if len(sys.argv) > 1 else 60.0
    rng = np.random.default_rng(int(sys.argv[2]) if len(sys.argv) > 2 else 2026)
    t0 = time.time(); n = bad = 0
    while time.time() - t0 < seconds:
        s = random_scene(rng)
        err = run_scene(s, rng, int(rng.integers(5, 60)))
        n += 1
        if err:
            bad += 1; print("MISMATCH", s.name, err[:600], flush=True)
        if n % 500 == 0:
            print(n, "scenes,", bad, "mismatches,", int(time.time() - t0), "s", flush=True)
    print("done:", n, "scenes,", bad, "mismatches")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
