"""Synthetic scene generators for the BASELINE.json configs (SURVEY.md §8d).

A scene is a plain bundle of numpy arrays in the reference's SoA layout (nudge.h:29-129): body
transforms / properties / momentum / idle counters, box and sphere colliders.  Body 0 is the static
world (example/main.cpp:391-395).  One collider per body, identity collider transform, collider tag =
collider index (+ box capacity for spheres) exactly as example/main.cpp:136-142,167-171 does.
Mass and inertia follow example/main.cpp:119-129 (boxes) and 154-160 (spheres).

Index-carrying fields are kept as uint32 here; `narrow()` helpers in the bindings cast them to the
reference's uint16 layout when a scene fits (<= 8192 colliders, <= 65535 bodies).
"""
import numpy as np

TRANSFORM = np.dtype([("position", "<f4", 3), ("body", "<u4"), ("rotation", "<f4", 4)], align=False)
PROPERTIES = np.dtype([("inertia_inverse", "<f4", 3), ("mass_inverse", "<f4")])
MOMENTUM = np.dtype([("velocity", "<f4", 3), ("unused0", "<f4"), ("angular_velocity", "<f4", 3), ("unused1", "<f4")])
BOX = np.dtype([("size", "<f4", 3), ("unused", "<f4")])
SPHERE = np.dtype([("radius", "<f4")])
CONTACT = np.dtype([("position", "<f4", 3), ("penetration", "<f4"), ("normal", "<f4", 3), ("friction", "<f4")])
IMPULSE = np.dtype([("impulse", "<f4", 3), ("unused", "<f4")])
PAIR16 = np.dtype([("a", "<u2"), ("b", "<u2")])
PAIR32 = np.dtype([("a", "<u4"), ("b", "<u4")])
# nb_ray / nb_ray_hit (include/nudge_b200.h): ray casts against the device-resident scene
RAY = np.dtype([("origin", "<f4", 3), ("max_t", "<f4"), ("direction", "<f4", 3), ("ignore_body", "<u4")])
RAY_HIT = np.dtype([("t", "<f4"), ("collider", "<u4"), ("body", "<u4"), ("tag", "<u4"), ("normal", "<f4", 3), ("unused", "<f4")])
NO_BODY = 0xFFFFFFFF

assert TRANSFORM.itemsize == 32 and MOMENTUM.itemsize == 32 and CONTACT.itemsize == 32
assert RAY.itemsize == 32 and RAY_HIT.itemsize == 32


def make_rays(origins, directions, max_t=np.inf, ignore_body=None):
    """A RAY array from [n, 3] origins and directions; max_t and ignore_body are scalars or [n] arrays (None: ignore no body)."""
    o = np.asarray(origins, np.float32).reshape(-1, 3)
    r = np.zeros(len(o), RAY)
    r["origin"] = o
    r["direction"] = np.asarray(directions, np.float32).reshape(-1, 3)
    r["max_t"] = max_t
    r["ignore_body"] = NO_BODY if ignore_body is None else ignore_body
    return r


class Scene:
    """Caller-owned simulation state (the arrays example/main.cpp:360-388 allocates)."""

    def __init__(self, n_bodies, n_boxes, n_spheres):
        self.transforms = np.zeros(n_bodies, TRANSFORM)
        self.transforms["rotation"][:, 3] = 1.0
        self.properties = np.zeros(n_bodies, PROPERTIES)
        self.momentum = np.zeros(n_bodies, MOMENTUM)
        self.idle = np.zeros(n_bodies, np.uint8)
        self.box_tags = np.zeros(n_boxes, np.uint32)
        self.box_data = np.zeros(n_boxes, BOX)
        self.box_transforms = np.zeros(n_boxes, TRANSFORM)
        self.box_transforms["rotation"][:, 3] = 1.0
        self.sphere_tags = np.zeros(n_spheres, np.uint32)
        self.sphere_data = np.zeros(n_spheres, SPHERE)
        self.sphere_transforms = np.zeros(n_spheres, TRANSFORM)
        self.sphere_transforms["rotation"][:, 3] = 1.0
        self.connections = np.zeros(0, PAIR32)
        # step parameters the reference leaves to the caller (example/main.cpp:275-305)
        self.time_step = np.float32(1.0 / 120.0)
        self.iterations = 8
        self.gravity = np.float32(9.82)
        self.damping = np.float32(0.25)
        self.name = "scene"

    @property
    def n_bodies(self):
        return len(self.transforms)

    @property
    def n_boxes(self):
        return len(self.box_tags)

    @property
    def n_spheres(self):
        return len(self.sphere_tags)

    @property
    def n_colliders(self):
        return self.n_boxes + self.n_spheres

    def copy(self):
        s = Scene(0, 0, 0)
        for k, v in self.__dict__.items():
            setattr(s, k, v.copy() if isinstance(v, np.ndarray) else v)
        return s

    def fits_reference(self):
        """True if the UNMODIFIED reference can run it (nudge.cpp:3010, uint16 indices nudge.h:68-71)."""
        return self.n_colliders <= 8192 and self.n_bodies <= 65535


def _box_props(size):
    """example/main.cpp:119-129, evaluated in float32 like the demo."""
    f = np.float32
    sx, sy, sz = size[:, 0].astype(f), size[:, 1].astype(f), size[:, 2].astype(f)
    mass = f(8.0) * sx * sy * sz
    k = mass * f(1.0 / 3.0)
    kx, ky, kz = k * sx * sx, k * sy * sy, k * sz * sz
    p = np.zeros(len(size), PROPERTIES)
    p["mass_inverse"] = f(1.0) / mass
    p["inertia_inverse"][:, 0] = f(1.0) / (ky + kz)
    p["inertia_inverse"][:, 1] = f(1.0) / (kx + kz)
    p["inertia_inverse"][:, 2] = f(1.0) / (kx + ky)
    return p


def _sphere_props(radius):
    """example/main.cpp:154-160."""
    f = np.float32
    r = radius.astype(f)
    mass = f(4.18879) * r * r * r
    k = f(2.5) / (mass * r * r)
    p = np.zeros(len(r), PROPERTIES)
    p["mass_inverse"] = f(1.0) / mass
    p["inertia_inverse"][:] = k[:, None]
    return p


def _random_unit_quaternions(rng, n):
    q = rng.normal(size=(n, 4)).astype(np.float32)
    q /= np.linalg.norm(q, axis=1, keepdims=True).astype(np.float32)
    return q.astype(np.float32)


def _assemble(name, box_sizes, box_pos, box_rot, radii, sph_pos, ground=True, ground_half=(400.0, 10.0, 400.0), ground_y=-20.0):
    """Body 0 static with an optional ground box (example/main.cpp:398-409), then one body per collider."""
    nb, ns = len(box_sizes), len(radii)
    g = 1 if ground else 0
    s = Scene(1 + nb + ns, g + nb, ns)
    s.name = name
    if ground:
        s.box_data["size"][0] = ground_half
        s.box_transforms["position"][0] = (0.0, ground_y, 0.0)
        s.box_transforms["body"][0] = 0
    s.box_tags[:] = np.arange(g + nb, dtype=np.uint32)
    s.box_data["size"][g:] = box_sizes
    s.box_transforms["body"][g:] = 1 + np.arange(nb, dtype=np.uint32)
    s.transforms["position"][1:1 + nb] = box_pos
    if box_rot is not None:
        s.transforms["rotation"][1:1 + nb] = box_rot
    s.properties[1:1 + nb] = _box_props(np.asarray(box_sizes, np.float32).reshape(-1, 3))
    # sphere tags are offset by the box capacity as in example/main.cpp:171
    s.sphere_tags[:] = np.arange(ns, dtype=np.uint32) + np.uint32(g + nb)
    s.sphere_data["radius"] = radii
    s.sphere_transforms["body"] = 1 + nb + np.arange(ns, dtype=np.uint32)
    s.transforms["position"][1 + nb:] = sph_pos
    s.properties[1 + nb:] = _sphere_props(np.asarray(radii, np.float32))
    return s


def demo_scene(n_boxes=1024, n_spheres=1024, iterations=8, seed=1, spread=5.0, height=300.0):
    """BASELINE config 0: ground + boxes + spheres falling (example/main.cpp:398-432), seeded PCG64."""
    rng = np.random.default_rng(seed)
    sizes = (rng.random((n_boxes, 3)) + 0.5).astype(np.float32)
    bpos = np.stack([rng.random(n_boxes) * 2 * spread - spread, rng.random(n_boxes) * height,
                     rng.random(n_boxes) * 2 * spread - spread], 1).astype(np.float32)
    radii = (rng.random(n_spheres) + 0.5).astype(np.float32)
    spos = np.stack([rng.random(n_spheres) * 2 * spread - spread, rng.random(n_spheres) * height,
                     rng.random(n_spheres) * 2 * spread - spread], 1).astype(np.float32)
    s = _assemble("demo_%db_%ds" % (n_boxes, n_spheres), sizes, bpos, None, radii, spos)
    s.iterations = iterations
    return s


def box_drop(n_boxes=65536, iterations=8, seed=2, density_L=None, spacing=(2.8, 2.6, 2.8), rotate=True):
    """BASELINE configs 1 and 3: N random boxes dropped onto the ground plane.

    Boxes start on a jittered lattice (random sizes U[0.5,1.5]^3 and random orientations) above a footprint of
    half-width L that keeps the survey probe's areal density (8191 boxes at L=15, SURVEY.md §8d), then fall and pile up."""
    rng = np.random.default_rng(seed)
    L = density_L if density_L is not None else 15.0 * np.sqrt(n_boxes / 8191.0)
    side = max(1, int(2 * L / spacing[0]))
    idx = rng.permutation(n_boxes)  # "random drop": body index carries no information about position
    layer, rem = idx // (side * side), idx % (side * side)
    gx, gz = rem // side, rem % side
    pos = np.stack([(gx + 0.5) * spacing[0] - L, layer * spacing[1] + 2.0, (gz + 0.5) * spacing[2] - L], 1)
    pos = (pos + rng.uniform(-0.2, 0.2, pos.shape)).astype(np.float32)
    sizes = (rng.random((n_boxes, 3)) + 0.5).astype(np.float32)
    rot = _random_unit_quaternions(rng, n_boxes) if rotate else None
    half = max(400.0, 2.0 * L)
    s = _assemble("box_drop_%d" % n_boxes, sizes, pos, rot, np.zeros(0, np.float32), np.zeros((0, 3), np.float32),
                  ground_half=(half, 10.0, half), ground_y=-10.0)
    s.iterations = iterations
    return s


def mixed_stack(n=262144, iterations=16, seed=3, jitter=0.05):
    """BASELINE config 2: 50/50 box/sphere lattice stack with small jitter (SURVEY.md §8d C3)."""
    rng = np.random.default_rng(seed)
    side = int(np.ceil((n / 8.0) ** 0.5))  # 8 layers
    idx = np.arange(n)
    layer, rem = idx // (side * side), idx % (side * side)
    gx, gz = rem // side, rem % side
    pos = np.stack([(gx - side / 2) * 2.2, layer * 2.2 + 1.2, (gz - side / 2) * 2.2], 1)
    pos = (pos + rng.uniform(-jitter, jitter, pos.shape)).astype(np.float32)
    is_box = (idx % 2) == 0
    nb = int(is_box.sum())
    sizes = np.full((nb, 3), 1.0, np.float32) * (0.8 + 0.2 * rng.random((nb, 1))).astype(np.float32)
    radii = (0.8 + 0.2 * rng.random(n - nb)).astype(np.float32)
    half = max(400.0, 2.5 * side)
    s = _assemble("mixed_stack_%d" % n, sizes, pos[is_box], None, radii, pos[~is_box], ground_half=(half, 10.0, half), ground_y=-10.0)
    s.iterations = iterations
    return s


def brick_wall(n=262144, iterations=20, width=None, gap=1e-3):
    """BASELINE config 4: running-bond wall of identical (1, 0.5, 0.5) half-extent bricks (SURVEY.md §8d C5)."""
    W = width if width is not None else int(np.ceil(np.sqrt(n * 2)))
    idx = np.arange(n)
    row, col = idx // W, idx % W
    x = (col - W / 2) * (2.0 + gap) + (row % 2) * 1.0
    y = row * (1.0 + gap) + 0.5 + gap
    pos = np.stack([x, y, np.zeros(n)], 1).astype(np.float32)
    sizes = np.tile(np.array([[1.0, 0.5, 0.5]], np.float32), (n, 1))
    half = max(400.0, 1.5 * W)
    s = _assemble("brick_wall_%d" % n, sizes, pos, None, np.zeros(0, np.float32), np.zeros((0, 3), np.float32),
                  ground_half=(half, 10.0, half), ground_y=-10.0)
    s.iterations = iterations
    return s


def two_boxes(pos_b=(0.0, 1.9, 0.0), rot_b=(0.0, 0.0, 0.0, 1.0), size_a=(1.0, 1.0, 1.0), size_b=(1.0, 1.0, 1.0)):
    """The shape of every reference unit test (tests/main.cpp:130-200): one box on static body 0, one on body 1."""
    s = Scene(2, 2, 0)
    s.name = "two_boxes"
    s.box_tags[:] = (0, 1)
    s.box_data["size"][0] = size_a
    s.box_data["size"][1] = size_b
    s.box_transforms["body"][:] = (0, 1)
    s.transforms["position"][1] = pos_b
    s.transforms["rotation"][1] = rot_b
    s.properties[1:] = _box_props(np.asarray([size_b], np.float32))
    return s


def hub_platform(n_side=55, iterations=4):
    """One DYNAMIC platform box carrying n_side^2 small boxes: every box-platform contact shares the platform's body, so the
    reference's batch scheduler (nudge.cpp:4206-4340) can never put two of them into one 8-lane batch.  Exercises the scheduler's
    open-slot list far beyond what a pile produces (the ADVICE.md hub-body case)."""
    n = n_side * n_side
    half = 0.6 * n_side + 2.0
    sizes = np.full((n + 1, 3), 0.5, np.float32); sizes[0] = (half, 1.0, half)
    pos = np.zeros((n + 1, 3), np.float32); pos[0] = (0.0, 5.0, 0.0)
    k = np.arange(n)
    pos[1:, 0] = (k % n_side - (n_side - 1) / 2.0) * 1.2
    pos[1:, 2] = (k // n_side - (n_side - 1) / 2.0) * 1.2
    pos[1:, 1] = 5.0 + 1.0 + 0.5 - 0.02
    s = _assemble("hub_platform_%d" % n, sizes, pos, None, np.zeros(0, np.float32), np.zeros((0, 3), np.float32))
    s.iterations = iterations
    return s
