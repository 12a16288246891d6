"""Known answers for the ray-cast restatement (oracle/raycast_ref.py), which the GPU tests hold nb_raycast to bit for bit.  CPU only."""
import numpy as np
from nudge_b200 import scenes as S
from oracle import raycast_ref as RR

f = np.float32


def _cast(s, origins, directions, max_t=np.inf, ignore_body=None):
    return RR.raycast_scene(s, S.make_rays(origins, directions, max_t, ignore_body))


def _boxes(positions, sizes, rotations=None):
    """Ground-less scene: body 0 static and empty, one box per body 1..n."""
    n = len(positions)
    s = S.Scene(n + 1, n, 0)
    s.box_tags[:] = 100 + np.arange(n)
    s.box_data["size"] = sizes
    s.box_transforms["body"] = 1 + np.arange(n)
    s.transforms["position"][1:] = positions
    if rotations is not None:
        s.transforms["rotation"][1:] = rotations
    return s


def test_ray_straight_down_onto_the_ground():
    s = S.demo_scene(4, 4, seed=3, height=300.0)      # ground: half extents (400, 10, 400) at y = -20, top face at y = -10
    h = _cast(s, [(1.5, -2.0, -2.25)], [(0.0, -1.0, 0.0)])[0]
    assert h["t"] == f(8.0) and h["collider"] == 0 and h["body"] == 0 and h["tag"] == s.box_tags[0]
    assert np.array_equal(h["normal"], np.array([0.0, 1.0, 0.0], f))
    h = _cast(s, [(1.5, -2.0, -2.25)], [(0.0, -0.5, 0.0)])[0]    # t counts units of the (non-unit) direction
    assert h["t"] == f(16.0)


def _rot64(q, v):
    u, w = q[..., :3], q[..., 3:4]
    return v + 2.0 * np.cross(u, np.cross(u, v) + w * v)


def test_rotated_boxes_and_spheres_against_float64():
    rng = np.random.default_rng(7)
    n = 64
    pos = rng.uniform(-20, 20, (n, 3)).astype(f)
    size = rng.uniform(0.3, 3.0, (n, 3)).astype(f)
    rot = S._random_unit_quaternions(rng, n)
    s = _boxes(pos, size, rot)
    # one ray per box from far outside, aimed near its centre; other boxes may be in the way, so compare against the float64 nearest hit
    dirs = rng.normal(size=(n, 3)); dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    aim = pos + rng.uniform(-0.2, 0.2, (n, 3)) * size
    origins = (aim - 60.0 * dirs).astype(f)
    dirs = (dirs * rng.uniform(0.5, 2.0, (n, 1))).astype(f)
    h = _cast(s, origins, dirs)
    o64, d64 = origins.astype(np.float64), dirs.astype(np.float64)
    q64 = rot.astype(np.float64); qc = q64 * np.array([-1, -1, -1, 1.0])
    t_best = np.full(n, np.inf); n_best = np.zeros((n, 3))
    for j in range(n):
        ol = _rot64(qc[j], o64 - pos[j].astype(np.float64)); dl = _rot64(qc[j], d64)
        s64 = size[j].astype(np.float64)
        with np.errstate(divide="ignore"):
            t1, t2 = (-s64 - ol) / dl, (s64 - ol) / dl
        tn, tf = np.minimum(t1, t2).max(1), np.maximum(t1, t2).min(1)
        ax = np.minimum(t1, t2).argmax(1)
        hit = (tn <= tf) & (tf >= 0) & (tn < t_best)
        t_best = np.where(hit, tn, t_best)
        nl = np.zeros((n, 3)); nl[np.arange(n), ax] = -np.sign(dl[np.arange(n), ax])
        n_best = np.where(hit[:, None], _rot64(q64[j], nl), n_best)
    assert np.isfinite(t_best).all() and (h["collider"] != S.NO_BODY).all()
    assert np.allclose(h["t"], t_best, rtol=1e-5, atol=0)
    assert np.allclose(h["normal"], n_best, atol=1e-4)

    # spheres: the quadratic in float64.  Origins a few radii away: b*b - a*c cancels (its float32 error grows with |m|^2 / r^2)
    m = 48
    c = rng.uniform(-20, 20, (m, 3)).astype(f); r = rng.uniform(0.3, 3.0, m).astype(f)
    s = S.Scene(m + 1, 0, m)
    s.sphere_tags[:] = np.arange(m); s.sphere_data["radius"] = r; s.sphere_transforms["body"] = 1 + np.arange(m)
    s.transforms["position"][1:] = c
    dirs = rng.normal(size=(m, 3)); dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    origins = (c + rng.uniform(-0.3, 0.3, (m, 3)) * r[:, None] - 4.0 * r[:, None] * dirs).astype(f)
    dirs = dirs.astype(f)
    h = _cast(s, origins, dirs)
    t_best = np.full(m, np.inf)
    for j in range(m):
        mm = origins.astype(np.float64) - c[j]; d64 = dirs.astype(np.float64)
        a = (d64 * d64).sum(1); b = (mm * d64).sum(1); cc = (mm * mm).sum(1) - float(r[j]) ** 2
        disc = b * b - a * cc
        with np.errstate(invalid="ignore"):
            t = np.where(cc <= 0, 0.0, (-b - np.sqrt(disc)) / a)
        ok = ((cc <= 0) | ((disc >= 0) & (t >= 0))) & (t < t_best)
        t_best = np.where(ok, t, t_best)
    hit = np.isfinite(t_best)
    assert hit.sum() > m // 2 and np.array_equal(h["collider"] != S.NO_BODY, hit)
    assert np.allclose(h["t"][hit], t_best[hit], rtol=1e-5, atol=0)
    out = hit & (h["t"] > 0)
    pts = origins[out].astype(np.float64) + h["t"][out, None] * dirs[out]
    want_n = (pts - c[h["collider"][out]]) / r[h["collider"][out], None]
    assert np.allclose(h["normal"][out], want_n, atol=1e-4) and not h["normal"][hit & ~out].any()


def test_origin_inside_a_collider():
    s = _boxes([(0.0, 0.0, 0.0)], [(1.0, 2.0, 3.0)], S._random_unit_quaternions(np.random.default_rng(1), 1))
    h = _cast(s, [(0.1, -0.2, 0.3)], [(1.0, 0.0, 0.0)])[0]
    assert h["t"] == 0.0 and h["collider"] == 0 and h["body"] == 1 and h["tag"] == 100 and not h["normal"].any()
    sp = S.demo_scene(0, 1, seed=2); sp.transforms["position"][1] = (5.0, 5.0, 5.0)
    h = _cast(sp, [(5.0, 5.0, 5.0)], [(0.0, 0.0, 0.0)])[0]      # a zero direction: only "inside" can hit
    assert h["t"] == 0.0 and h["collider"] == 1 and not h["normal"].any()


def test_zero_direction_components():
    s = _boxes([(0.0, 0.0, 0.0)], [(1.0, 1.0, 1.0)])
    edge = f(1.0); outside = np.nextafter(edge, f(2.0))
    h = _cast(s, [(edge, 5.0, 0.0), (outside, 5.0, 0.0), (0.0, 5.0, -edge), (0.0, 5.0, -outside)], [(0.0, -1.0, 0.0)] * 4)
    assert list(h["collider"]) == [0, S.NO_BODY, 0, S.NO_BODY]
    assert h["t"][0] == 4.0 and np.array_equal(h["normal"][0], np.array([0.0, 1.0, 0.0], f))
    assert h["t"][1] == np.inf and not h["normal"][1].any()


def test_max_t_cutoff_on_each_side_of_the_hit():
    rng = np.random.default_rng(3)
    s = _boxes([(0.0, 0.0, 0.0)], [(1.0, 0.7, 1.3)], S._random_unit_quaternions(rng, 1))
    ray = [(0.3, 10.0, -0.2)], [(0.01, -1.0, 0.02)]
    t = _cast(s, *ray)[0]["t"]
    assert 0 < t < np.inf
    below, above = np.nextafter(t, f(0.0)), np.nextafter(t, f(np.inf))
    h = _cast(s, ray[0] * 3, ray[1] * 3, max_t=np.array([below, t, above], f))
    assert list(h["collider"]) == [S.NO_BODY, 0, 0]
    assert h["t"][0] == below and h["t"][1] == t and h["t"][2] == t


def test_ignore_body():
    s = S.demo_scene(1, 0, seed=4)                    # ground (body 0) and one box on body 1
    s.transforms["position"][1] = (0.0, 0.0, 0.0)
    o, d = [(0.0, 20.0, 0.0)], [(0.0, -1.0, 0.0)]
    assert _cast(s, o, d)[0]["body"] == 1
    h = _cast(s, o, d, ignore_body=1)[0]
    assert h["body"] == 0 and h["collider"] == 0 and h["t"] == 30.0
    assert _cast(s, o, d, ignore_body=0)[0]["body"] == 1
    h = _cast(s, o * 2, d * 2, ignore_body=np.array([0, 1], np.uint32))
    assert list(h["body"]) == [1, 0]


def test_coincident_boxes_go_to_the_lower_index():
    s = _boxes([(0.0, 0.0, 0.0)] * 3, [(1.0, 1.0, 1.0)] * 3)
    h = _cast(s, [(0.2, 5.0, 0.1), (0.0, 0.0, 0.0)], [(0.0, -1.0, 0.0), (0.0, 1.0, 0.0)])
    assert list(h["collider"]) == [0, 0] and list(h["tag"]) == [100, 100] and h["t"][0] == 4.0
    h = _cast(s, [(0.2, 5.0, 0.1)], [(0.0, -1.0, 0.0)], ignore_body=1)[0]
    assert h["collider"] == 1 and h["body"] == 2


def test_world_transforms_restate_the_collision_stage():
    """collider_world is the collision stage's body * collider (the step's oracle computes the same): off-centre rotated colliders."""
    rng = np.random.default_rng(9)
    s = S.demo_scene(20, 10, seed=5)
    s.transforms["rotation"][1:] = S._random_unit_quaternions(rng, s.n_bodies - 1)
    s.box_transforms["position"][1:] = rng.normal(size=(s.n_boxes - 1, 3)).astype(f)
    s.box_transforms["rotation"][1:] = S._random_unit_quaternions(rng, s.n_boxes - 1)
    w = RR.collider_world(s.transforms, s.box_transforms, s.sphere_transforms).astype([(n, s.transforms.dtype[n]) for n in s.transforms.dtype.names])
    cx = np.concatenate([s.box_transforms, s.sphere_transforms]); b = s.transforms[cx["body"]]
    want = b["position"].astype(np.float64) + _rot64(b["rotation"].astype(np.float64), cx["position"].astype(np.float64))
    assert np.abs(w["position"] - want).max() < 1e-4 and np.array_equal(w["body"], cx["body"])
