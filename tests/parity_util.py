"""Stage-by-stage bit comparison helpers shared by the CPU (oracle vs reference) and GPU (CUDA vs oracle) parity tests."""
import hashlib
import numpy as np
from nudge_b200 import abi


def bits(a):
    return np.ascontiguousarray(a).view(np.uint8)


class Report:
    def __init__(self, label=""):
        self.label = label
        self.failures = []

    def eq(self, name, x, y):
        x = np.asarray(x); y = np.asarray(y)
        ok = x.shape == y.shape and x.dtype.itemsize == y.dtype.itemsize and np.array_equal(bits(x), bits(y))
        if not ok:
            msg = "%s %s: shapes %s vs %s" % (self.label, name, x.shape, y.shape)
            if x.shape == y.shape and len(x):
                xv = bits(x).reshape(len(x), -1); yv = bits(y).reshape(len(y), -1)
                bad = np.nonzero((xv != yv).any(axis=1))[0]
                msg += "; %d/%d rows differ, first %s\n   want %s\n   got  %s" % (len(bad), len(x), bad[:4], x[bad[0]], y[bad[0]])
            self.failures.append(msg)
        return ok

    def check(self, name, cond, detail=""):
        if not cond:
            self.failures.append("%s %s %s" % (self.label, name, detail))
        return cond

    @property
    def ok(self):
        return not self.failures

    def __str__(self):
        return "\n".join(self.failures) if self.failures else "OK"


def rows_by_contact(view, n_contacts):
    """Reference / oracle store rows per batch lane; key them by contact (first lane of a duplicated contact)."""
    lanes = len(view["contact"])
    first = np.full(n_contacts, lanes, np.int64)
    np.minimum.at(first, view["contact"].astype(np.int64), np.arange(lanes))
    assert (first < lanes).all()
    return dict(rows=view["rows"][first], states=view["states"][first], batch=(first // 8).astype(np.uint32), slot=first.astype(np.uint32),
                a=view["a"][first], b=view["b"][first])


def ref_layout_stages(x, widened):
    """Runs one full step of x (the reference's RefSim, or the widened OracleSim with widened=True) and yields (stage, array) after every
    stage, each array in the reference's uint16 / packed-tag layout, so that the two implementations, or one of them and digests of the
    other recorded earlier (tests/golden/make_ref_traces.py), compare byte for byte."""
    tag = (lambda v, t, f: abi.wide_tag_to_ref(v[t], v[f])) if widened else (lambda v, t, f: v[t])
    u32 = lambda a: np.asarray(a).astype(np.uint32)
    x.collide()
    c = x.contacts_view()
    yield "contact count", np.array([c["count"]], np.uint32)
    yield "active", u32(c["active"])
    yield "contacts", c["data"]
    yield "bodies.a", u32(c["bodies"]["a"])
    yield "bodies.b", u32(c["bodies"]["b"])
    yield "tags", tag(c, "tags", "features")
    yield "sleeping", abi.wide_pair_to_ref(c["sleeping"]) if widened else c["sleeping"]
    x.apply_gravity_damping()
    yield "momentum after gravity", x.momentum
    x.read_cached_impulses()
    i = x.impulses_view()
    yield "sorted", i["sorted"]
    yield "impulses", i["data"]
    yield "culled tags", tag(i, "culled_tags", "culled_features")
    yield "culled data", i["culled_data"]
    x.setup_contact_constraints()
    k = x.constraints_view()
    yield "batches", np.array([k["batches"]], np.uint32)
    yield "constraint_to_contact", k["contact"]
    yield "rows", k["rows"]
    yield "warm-start states", k["states"]
    yield "momentum after setup", x.momentum
    for it in range(int(x.scene.iterations)):
        x.apply_impulses()
        yield "momentum sweep %d" % it, x.momentum
    yield "states", x.constraints_view()["states"]
    x.update_cached_impulses()
    yield "updated impulses", x.impulses_view()["data"]
    x.write_cached_impulses()
    cv = x.cache_view()
    yield "cache tags", tag(cv, "tags", "features")
    yield "cache data", cv["data"]
    x.advance()
    yield "transforms", x.transforms
    yield "idle", x.idle


# stages after which a difference makes the rest of the step meaningless to compare (array lengths follow from them)
_STOP_AFTER = ("contact count", "sleeping", "batches")


def compare_ref_oracle_step(r, o, rep):
    """One full step, the unmodified reference (uint16 layout) against the widened restatement."""
    for (name, a), (_, b) in zip(ref_layout_stages(r, False), ref_layout_stages(o, True)):
        rep.eq(name, a, b)
        if name in _STOP_AFTER and not rep.ok:
            return False
    return rep.ok


def stage_digest(a):
    """8-byte digest of an array's shape and bytes: what the golden reference traces store per stage."""
    h = hashlib.blake2b(digest_size=8)
    h.update(repr(np.shape(a)).encode())
    h.update(bits(a).tobytes())
    return np.frombuffer(h.digest(), np.uint64)[0]


def compare_oracle_gpu_step(o, g, rep, sweeps_individually=True):
    """One full step, the widened CPU oracle against the CUDA path, every stage bit for bit.  Both must start from the same state."""
    o.collide(); g.collide()
    g.download_contacts()
    oc, gc = o.contacts_view(), g.contacts_view()
    op, gp = o.pairs_view(), g.pairs_view()
    rep.eq("morton order", op["order"], gp["order"])
    rep.eq("pairs.lo", op["lo"], gp["lo"]); rep.eq("pairs.hi", op["hi"], gp["hi"])
    rep.check("contact count", oc["count"] == gc["count"], "%d vs %d" % (oc["count"], gc["count"]))
    rep.eq("active", oc["active"], gc["active"])
    if oc["count"] != gc["count"]:
        return False
    rep.eq("contacts", oc["data"], gc["data"]); rep.eq("bodies", oc["bodies"], gc["bodies"])
    rep.eq("tags", oc["tags"], gc["tags"]); rep.eq("features", oc["features"], gc["features"])
    rep.eq("sleeping", oc["sleeping"], gc["sleeping"])
    if not rep.ok:
        return False
    n = oc["count"]
    o.apply_gravity_damping(); g.apply_gravity_damping()
    g.download_bodies()
    rep.eq("momentum after gravity", o.momentum, g.momentum)
    o.read_cached_impulses(); g.read_cached_impulses()
    oi, gi = o.impulses_view(), g.impulses_view()
    rep.eq("sorted", oi["sorted"], gi["sorted"]); rep.eq("impulses", oi["data"], gi["data"])
    rep.eq("culled tags", oi["culled_tags"], gi["culled_tags"]); rep.eq("culled features", oi["culled_features"], gi["culled_features"])
    rep.eq("culled data", oi["culled_data"], gi["culled_data"])
    o.setup_contact_constraints(); g.setup_contact_constraints()
    ok_, gk = rows_by_contact(o.constraints_view(), n), g.constraints_view()
    order = gk["contact"].astype(np.int64)
    if n:
        rep.check("row contacts are a permutation", len(order) == n and np.array_equal(np.sort(order), np.arange(n)))
        rep.eq("batch index", ok_["batch"], gk["batch_of_contact"])
        rep.eq("slot (batch*8 + lane)", ok_["slot"], gk["slot_of_contact"])
        rep.eq("rows", ok_["rows"][order], gk["rows"]); rep.eq("row a", ok_["a"][order], gk["a"]); rep.eq("row b", ok_["b"][order], gk["b"])
        rep.eq("warm-start states", ok_["states"][order], gk["states"])
    g.download_bodies()
    rep.eq("momentum after setup", o.momentum, g.momentum)
    if not rep.ok:
        return False
    its = int(o.scene.iterations)
    if sweeps_individually:
        for it in range(its):
            o.apply_impulses(); g.apply_impulses(1)
            g.download_bodies()
            rep.eq("momentum sweep %d" % it, o.momentum, g.momentum)
    else:
        for it in range(its):
            o.apply_impulses()
        g.apply_impulses(its)
        g.download_bodies()
        rep.eq("momentum after %d sweeps" % its, o.momentum, g.momentum)
    if n:
        rep.eq("states", rows_by_contact(o.constraints_view(), n)["states"][order], g.constraints_view()["states"])
    o.update_cached_impulses(); g.update_cached_impulses()
    rep.eq("updated impulses", o.impulses_view()["data"], g.impulses_view()["data"])
    o.write_cached_impulses(); g.write_cached_impulses()
    g.download_cache()
    ocv, gcv = o.cache_view(), g.cache_view()
    rep.eq("cache tags", ocv["tags"], gcv["tags"]); rep.eq("cache features", ocv["features"], gcv["features"]); rep.eq("cache data", ocv["data"], gcv["data"])
    o.advance(); g.advance()
    g.download_bodies()
    rep.eq("transforms", o.transforms, g.transforms); rep.eq("idle", o.idle, g.idle)
    return rep.ok


def sync_oracle_from_gpu(o, g):
    """Copies the GPU simulation's body state and contact cache into an oracle instance (same Scene), so that one
    step can be compared from identical input state (SURVEY.md §0.6: never compare long trajectories)."""
    g.download_bodies(); g.download_cache()
    o.transforms[:] = g.transforms; o.momentum[:] = g.momentum; o.idle[:] = g.idle
    n = g.cache.count
    o.cache_tags[:n] = g.cache_tags[:n]; o.cache_features[:n] = g.cache_features[:n]; o.cache_data[:n] = g.cache_data[:n]
    o.cache.count = n
