import os
import numpy as np
from nudge_b200 import scenes as S, abi

HERE = os.path.dirname(os.path.abspath(__file__))


def load_box_cases():
    return np.load(os.path.join(HERE, "golden", "box_box_cases.npz"))


def scene_of(g, k):
    s = S.Scene(2, 2, 0)
    s.box_tags[:] = (0, 1)
    s.box_data["size"][:] = g["size"][k]
    s.box_transforms["position"][:] = g["cpos"][k]
    s.box_transforms["rotation"][:] = g["crot"][k]
    s.box_transforms["body"][:] = g["cbody"][k]
    s.transforms["position"][1] = g["bpos"][k]; s.transforms["rotation"][1] = g["brot"][k]
    return s


def check_case(g, k, view):
    """view: contacts_view() of a widened implementation.  Returns an error string or None."""
    m = int(g["count"][k])
    if view["count"] != m:
        return "case %d family %d: %d contacts, reference has %d" % (k, g["family"][k], view["count"], m)
    if m != int(g["expect"][k]):
        return "case %d: fixture disagrees with the reference test's expected count" % k
    if not np.array_equal(view["data"].view(np.uint8), g["contacts"][k, :m].view(np.uint8)):
        return "case %d family %d: contact data differs" % (k, g["family"][k])
    if not (np.array_equal(view["bodies"]["a"], g["bodies"][k, :m, 0]) and np.array_equal(view["bodies"]["b"], g["bodies"][k, :m, 1])):
        return "case %d: bodies differ" % k
    if not np.array_equal(abi.wide_tag_to_ref(view["tags"], view["features"]), g["tags"][k, :m]):
        return "case %d family %d: tags differ" % (k, g["family"][k])
    return None


# ---- the reference's own demo application, recorded headless (tests/golden/make_demo_golden.py, oracle/demo_capture.cpp) ----
def load_demo_frames():
    return np.load(os.path.join(HERE, "golden", "demo_frames.npz"))


def demo_scene(g, state="initial"):
    """The demo's scene (example/main.cpp:391-432: ground + 1024 boxes + 512 spheres from rand()) with the body state of `state`
    ("initial" = before the first simulate(), "f0", "f40" = recorded frames) and the demo's step parameters (example/main.cpp:274-305)."""
    nb, nbox, nsph = len(g["initial_transforms"]), len(g["initial_box_tags"]), len(g["initial_sphere_tags"])
    s = S.Scene(nb, nbox, nsph)
    s.transforms[:] = np.ascontiguousarray(g[state + "_transforms"]).view(S.TRANSFORM).reshape(nb)
    s.momentum[:] = np.ascontiguousarray(g[state + "_momentum"]).view(S.MOMENTUM).reshape(nb)
    s.idle[:] = g[state + "_idle"]
    s.properties[:] = np.ascontiguousarray(g["initial_properties"]).view(S.PROPERTIES).reshape(nb)
    s.box_transforms[:] = np.ascontiguousarray(g["initial_box_transforms"]).view(S.TRANSFORM).reshape(nbox)
    s.box_data[:] = np.ascontiguousarray(g["initial_box_data"]).view(S.BOX).reshape(nbox)
    s.box_tags[:] = g["initial_box_tags"]
    s.sphere_transforms[:] = np.ascontiguousarray(g["initial_sphere_transforms"]).view(S.TRANSFORM).reshape(nsph)
    s.sphere_data["radius"][:] = g["initial_sphere_data"]
    s.sphere_tags[:] = g["initial_sphere_tags"]
    s.time_step = np.float32(1.0 / (60.0 * 2.0)); s.iterations = 20; s.gravity = np.float32(9.82); s.damping = np.float32(0.25)
    s.name = "reference demo (recorded)"
    return s


def demo_substeps(frame):
    """simulate() calls behind recorded frame f: f + 1, two sub-steps each (example/main.cpp:275, 330-334)."""
    return 2 * (frame + 1)


# ---- every stage of every step of the reference, as digests (tests/golden/make_ref_traces.py, parity_util.ref_layout_stages) ----
def load_ref_traces():
    return np.load(os.path.join(HERE, "golden", "ref_traces.npz"))


def _sleep_after(step, seed, share):
    """Hook: before `step`, put a seeded random `share` of the bodies to sleep (idle counter 0xff, momentum zeroed)."""
    def hook(i, sim):
        if i == step:
            m = np.random.default_rng(seed).random(sim.scene.n_bodies) < share
            sim.idle[m] = 0xff
            sim.momentum["velocity"][m] = 0; sim.momentum["angular_velocity"][m] = 0
    return hook


def ref_trace_cases(name):
    """Yields (case, scene, steps, contact capacity, hook(i, sim) run before step i) for the traces of test_oracle_vs_ref.py's `name`.
    The fuzz cases share one generator and must be run in order, each to the end, before the next is drawn."""
    cap = lambda s: max(1024, 64 * s.n_bodies)
    if name == "small_mixed":
        s = S.demo_scene(100, 100, iterations=4, spread=2.0, height=20.0); yield name, s, 30, cap(s), None
    elif name == "demo_config0":
        s = S.demo_scene(1024, 1024, iterations=8); yield name, s, 4, cap(s), None
    elif name == "rotated_box_drop":
        s = S.box_drop(1500, iterations=8); yield name, s, 12, cap(s), None
    elif name == "sleeping_islands":
        s = S.demo_scene(120, 120, iterations=4, spread=6.0, height=6.0, seed=11); yield name, s, 46, cap(s), _sleep_after(40, 5, 0.8)
    elif name == "fuzz":
        from tests import fuzz_oracle_vs_ref as F
        rng = np.random.default_rng(77)
        for k in range(120):
            s = F.random_scene(rng)
            yield "fuzz%03d" % k, s, int(rng.integers(5, 40)), F.contact_capacity(s), (lambda i, sim: F.maybe_sleep(rng, (sim,)))
    else:
        raise KeyError(name)
