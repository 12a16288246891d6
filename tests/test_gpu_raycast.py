"""Ray casts against the device-resident scene (nb_build_query_tree / nb_raycast): bit-identical to the brute-force float32 restatement
(oracle/raycast_ref.py) whatever the tree prunes, the step untouched by queries, snapshot semantics and argument errors."""
import ctypes as C
import numpy as np
import pytest
import nudge_b200
from nudge_b200 import scenes, abi
from oracle import raycast_ref as RR

pytestmark = pytest.mark.gpu

f = np.float32
NB_ERR_ARGUMENT = -3


def _bits(h):
    return np.ascontiguousarray(h).view(np.uint32).reshape(-1, 8)


def _assert_hits_equal(got, want, what):
    bad = (_bits(got) != _bits(want)).any(1)
    assert not bad.any(), "%s: %d of %d rays differ, first %d: got %r want %r" % (what, bad.sum(), len(got), np.argmax(bad), got[np.argmax(bad)], want[np.argmax(bad)])


def _demo_after_steps():
    s = scenes.demo_scene(1024, 1024, iterations=8)
    sim = nudge_b200.Sim(s)
    for _ in range(200):
        sim.step()
    return sim


def _offcentre_scene():
    """The scene of test_gpu_render: colliders off their bodies' centres and rotated against them."""
    import torch
    rng = np.random.default_rng(11)
    s = scenes.demo_scene(700, 333, iterations=8, spread=5.0, height=40.0)
    s.box_transforms["position"][1:] = rng.normal(size=(s.n_boxes - 1, 3)).astype(f) * 0.2
    s.box_transforms["rotation"][1:] = scenes._random_unit_quaternions(rng, s.n_boxes - 1)
    s.sphere_transforms["position"][:] = rng.normal(size=(s.n_spheres, 3)).astype(f) * 0.2
    side = torch.cuda.Stream()
    sim = nudge_b200.Sim(s, stream=side.cuda_stream)
    sim._keep_stream = side
    for _ in range(25):
        sim.step()
    return sim


def _adversarial_rays(sim, rng, n_random=10000):
    """Random rays plus rays aimed exactly at box corners and edge midpoints, axis-parallel rays with zero components and origins
    inside colliders."""
    w = RR.collider_world(sim.transforms, sim.box_transforms, sim.sphere_transforms)
    pos = w["position"].astype(np.float64)
    lo, hi = pos.min(0) - 5.0, pos.max(0) + 5.0
    out = []
    o = rng.uniform(lo, hi, (n_random, 3)).astype(f)
    d = (rng.normal(size=(n_random, 3)) * rng.uniform(0.25, 4.0, (n_random, 1))).astype(f)
    out.append(scenes.make_rays(o, d))
    # corners and edge midpoints of boxes (float64 world points rounded to float32; the ray passes through them to float precision)
    nb = sim.scene.n_boxes
    pick = rng.choice(np.arange(1, nb), min(300, nb - 1), replace=False)
    signs = np.array([[sx, sy, sz] for sx in (-1, 1) for sy in (-1, 1) for sz in (-1, 1)], np.float64)
    mids = np.array([[0, sy, sz] for sy in (-1, 1) for sz in (-1, 1)] + [[sx, 0, sz] for sx in (-1, 1) for sz in (-1, 1)] +
                    [[sx, sy, 0] for sx in (-1, 1) for sy in (-1, 1)], np.float64)
    q = w["rotation"][pick].astype(np.float64)
    size = sim.box_data["size"][pick].astype(np.float64)
    for local in (signs, mids):
        pts = pos[pick, None, :] + _rot64(q[:, None, :], local[None, :, :] * size[:, None, :])
        pts = pts.reshape(-1, 3)
        away = rng.normal(size=pts.shape); away /= np.linalg.norm(away, axis=1, keepdims=True)
        org = (pts + 6.0 * away).astype(f)
        out.append(scenes.make_rays(org, (pts - org).astype(f)))
    # axis-parallel rays (two zero direction components), from random points and from exactly above corners
    k = 3000
    axis = rng.integers(0, 3, k); sgn = rng.choice([-1.0, 1.0], k)
    d = np.zeros((k, 3), f); d[np.arange(k), axis] = sgn
    out.append(scenes.make_rays(rng.uniform(lo, hi, (k, 3)).astype(f), d))
    corners = (pos[pick, None, :] + _rot64(q[:, None, :], signs[None] * size[:, None, :])).reshape(-1, 3).astype(f)
    org = corners.copy(); org[:, 1] += f(10.0)
    out.append(scenes.make_rays(org, np.tile(np.array([[0.0, -1.0, 0.0]], f), (len(org), 1))))
    # origins inside colliders (centres and just inside)
    inside = rng.choice(len(w), 500, replace=False)
    out.append(scenes.make_rays(w["position"][inside], rng.normal(size=(500, 3)).astype(f)))
    return np.concatenate(out)


def _rot64(q, v):
    u, s = q[..., :3], q[..., 3:4]
    return v + 2.0 * np.cross(u, np.cross(u, v) + s * v)


@pytest.mark.parametrize("make", [_demo_after_steps, _offcentre_scene], ids=["demo_200_steps", "offcentre_rotated"])
def test_bit_identical_to_the_oracle(make):
    sim = make()
    sim.download_bodies()
    rng = np.random.default_rng(5)
    rays = _adversarial_rays(sim, rng)
    sim.build_query_tree()
    got = sim.raycast(rays=rays)
    want = RR.raycast_scene(sim, rays)
    assert (want["collider"] != scenes.NO_BODY).sum() > len(rays) // 4
    _assert_hits_equal(got, want, "random + adversarial rays")
    # max_t one ulp below / at / above the true hit, ignore_body = the hit body and 0
    hit = np.nonzero((want["collider"] != scenes.NO_BODY) & (want["t"] > 0))[0][:3000]
    base = rays[hit]
    t = want["t"][hit]
    sets = []
    for mt in (np.nextafter(t, f(0.0)), t, np.nextafter(t, f(np.inf))):
        r = base.copy(); r["max_t"] = mt; sets.append(r)
    for ib in (want["body"][hit], np.zeros(len(hit), np.uint32)):
        r = base.copy(); r["ignore_body"] = ib; sets.append(r)
    more = np.concatenate(sets)
    got = sim.raycast(rays=more)
    want2 = RR.raycast_scene(sim, more)
    n = len(hit)
    assert (want2["collider"][:n] == scenes.NO_BODY).all() and np.array_equal(want2["collider"][n:3 * n], np.tile(want["collider"][hit], 2))
    _assert_hits_equal(got, want2, "max_t / ignore_body rays")


def test_settled_pile_at_scale_through_torch_tensors():
    import torch
    side = torch.cuda.Stream()
    s = scenes.box_drop(65536, iterations=8, seed=2)
    sim = nudge_b200.Sim(s, stream=side.cuda_stream)
    for _ in range(600):
        sim.step()
    sim.download_bodies()
    assert sim.counts().overflow == 0
    rng = np.random.default_rng(8)
    n = 1 << 20
    pos = sim.transforms["position"][1:]
    lo, hi = pos.min(0), pos.max(0)
    o = rng.uniform(lo, hi, (n, 3)).astype(f)
    o[: n // 2, 1] = hi[1] + 5.0
    d = rng.normal(size=(n, 3)).astype(f)
    d[: n // 2] = (0.0, -1.0, 0.0)
    d[: n // 2, 0] = rng.normal(size=n // 2) * 0.05
    rays = scenes.make_rays(o, d)
    with torch.cuda.stream(side):
        r_dev = torch.from_numpy(rays.view(np.int32).reshape(n, 8)).cuda()
        h_dev = torch.empty((n, 8), dtype=torch.int32, device="cuda")
        sim.build_query_tree()
        sim.raycast(device_ptr=r_dev.data_ptr(), hits_ptr=h_dev.data_ptr(), n=n)
        perm = torch.from_numpy(rng.permutation(n)).cuda()
        r_perm = r_dev[perm].contiguous()
        h_perm = torch.empty_like(h_dev)
        sim.raycast(device_ptr=r_perm.data_ptr(), hits_ptr=h_perm.data_ptr(), n=n)
    side.synchronize()
    hits = h_dev.cpu().numpy().view(scenes.RAY_HIT).reshape(n)
    assert np.array_equal(h_perm.cpu().numpy(), h_dev[perm].cpu().numpy())
    assert (hits["collider"] != scenes.NO_BODY).mean() > 0.5
    sub = rng.choice(n, 8192, replace=False)
    want = RR.raycast_scene(sim, rays[sub], parallel=True)
    _assert_hits_equal(hits[sub], want, "8192-ray subset of the settled pile")


def _state(sim):
    sim.download_bodies()
    c = sim.counts()
    return (sim.transforms.copy(), sim.momentum.copy(), sim.idle.copy(), tuple(getattr(c, k) for k, _ in c._fields_))


def _probe_rays(rng, n=4096):
    return scenes.make_rays(rng.uniform(-8, 8, (n, 3)).astype(f) + f([0, 6, 0]), rng.normal(size=(n, 3)).astype(f))


def test_the_step_is_untouched_by_queries():
    """N steps with a build and a raycast between every step (graph path) or between every pair of the seven stage calls give the
    bits of the same N steps without queries.  The scene is a lattice drop (no initial overlap) that lands during the run, so contacts,
    islands and the warm-started cache are all on the path; two query-free runs must agree first, or the comparison would mean nothing."""
    import torch
    s = scenes.box_drop(4096, iterations=8, seed=3)
    rng = np.random.default_rng(2)
    rays = scenes.make_rays(rng.uniform(-12, 12, (4096, 3)).astype(f) + f([0, 8, 0]), rng.normal(size=(4096, 3)).astype(f))
    steps = 150

    def graph_run(query):
        side = torch.cuda.Stream()
        sim = nudge_b200.Sim(s, stream=side.cuda_stream)
        for _ in range(steps):
            sim.step()
            if query:
                sim.build_query_tree(); sim.raycast(rays=rays)
        st = _state(sim)
        assert sim.debug_scalar("graph_coop") != 0, "the step was expected on the CUDA-graph path"
        sim.close()
        return st

    def staged_run(query):
        sim = nudge_b200.Sim(s)
        calls = [sim.collide, sim.apply_gravity_damping, sim.read_cached_impulses, sim.setup_contact_constraints,
                 lambda: sim.apply_impulses(int(s.iterations)), sim.update_cached_impulses, sim.write_cached_impulses, sim.advance]
        for _ in range(steps):
            for c in calls:
                c()
                if query:
                    sim.build_query_tree(); sim.raycast(rays=rays)
        st = _state(sim)
        sim.close()
        return st

    for run in (graph_run, staged_run):
        a, a2, b = run(False), run(False), run(True)
        assert a[3][2] > 1000, "the boxes were expected to be in contact by the end of the run"
        for x, y in zip(a[:3], a2[:3]):
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), "%s: the step is not reproducible on this scene" % run.__name__
        for x, y in zip(a[:3], b[:3]):
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), "%s: queries changed the step" % run.__name__
        assert a[3] == a2[3] == b[3]


def test_snapshot_semantics():
    s = scenes.demo_scene(300, 300, iterations=8, spread=3.0, height=30.0)
    sim = nudge_b200.Sim(s)
    for _ in range(20):
        sim.step()
    sim.build_query_tree()
    q = sim.debug("query_world_xf", np.uint32)
    sim.collide()
    w = sim.debug("world_xf", np.uint32)
    assert len(q) == 8 * s.n_colliders and np.array_equal(q, w)
    sim.download_bodies()
    wq = RR.collider_world(sim.transforms, sim.box_transforms, sim.sphere_transforms)
    assert np.array_equal(wq.view(np.uint32), q)
    rays = _probe_rays(np.random.default_rng(4))
    rays["origin"][:, 1] += f(15.0)
    before = sim.raycast(rays=rays)
    _assert_hits_equal(before, RR.raycast_scene(sim, rays), "snapshot")
    moved = sim.transforms.copy()
    for _ in range(20):
        sim.step()                         # bodies are still falling: the scene moves, the snapshot does not
    sim.download_bodies()
    assert not np.array_equal(moved, sim.transforms)
    _assert_hits_equal(sim.raycast(rays=rays), before, "rays after nb_step without a rebuild")
    sim.build_query_tree()
    after = sim.raycast(rays=rays)
    _assert_hits_equal(after, RR.raycast_scene(sim, rays), "rebuilt snapshot")
    assert not np.array_equal(_bits(after), _bits(before))


def test_errors():
    big = scenes.demo_scene(64, 64)
    sim = nudge_b200.Sim(big)
    lib, ctx, st = sim.lib, sim.ctx, sim.stream
    rays = scenes.make_rays([(0.0, 5.0, 0.0)], [(0.0, -1.0, 0.0)])
    hits = np.zeros(1, scenes.RAY_HIT)
    assert lib.nb_raycast(ctx, abi.ptr(rays), abi.ptr(hits), 1, 0, st) == NB_ERR_ARGUMENT      # no snapshot yet
    sim.build_query_tree()
    assert lib.nb_raycast(ctx, abi.ptr(rays), abi.ptr(hits), 1, 0, st) == 0 and hits["collider"][0] != scenes.NO_BODY
    assert lib.nb_raycast(ctx, None, None, 0, 0, st) == 0 and lib.nb_raycast(ctx, None, None, 0, 1, st) == 0   # n = 0
    assert lib.nb_raycast(ctx, None, abi.ptr(hits), 1, 0, st) == NB_ERR_ARGUMENT
    assert lib.nb_raycast(ctx, abi.ptr(rays), None, 1, 0, st) == NB_ERR_ARGUMENT
    assert lib.nb_raycast(ctx, None, None, 1, 1, st) == NB_ERR_ARGUMENT
    sim.reload(scenes.demo_scene(32, 16))          # nb_upload_colliders with other counts: the snapshot no longer fits
    assert lib.nb_raycast(ctx, abi.ptr(rays), abi.ptr(hits), 1, 0, st) == NB_ERR_ARGUMENT
    assert lib.nb_raycast(ctx, abi.ptr(rays), abi.ptr(hits), 1, 0, st) == NB_ERR_ARGUMENT
    sim.build_query_tree()
    assert lib.nb_raycast(ctx, abi.ptr(rays), abi.ptr(hits), 1, 0, st) == 0
    with pytest.raises(nudge_b200.NudgeError):
        nudge_b200.Sim(big).raycast([(0.0, 0.0, 0.0)], [(0.0, 1.0, 0.0)])
    empty = nudge_b200.Sim(scenes.demo_scene(64, 64))
    empty.build_query_tree()
    h = empty.raycast(np.zeros((0, 3), f), np.zeros((0, 3), f))
    assert len(h) == 0
