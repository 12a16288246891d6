"""CPU restatement of the ray casts (nb_build_query_tree / nb_raycast; TEST INFRASTRUCTURE ONLY, tests/ imports it).

Brute force over every collider, no tree: float32 throughout, one IEEE operation per kernel operation in the kernel's order (the library is
built with -fmad=false -prec-div=true -prec-sqrt=true), so the result is bit-comparable with nudge_b200/csrc/nb_query_api.cuh.  The operation
order is the one DESIGN.md section 8.5 fixes:

  collider world transform (k_collider_world): p = qrot(body.q, collider.p) + body.p, q = qmul(body.q, collider.q), where
      qrot(q, r) = (r + q.w * t) + cross(q.v, t) with t = 2 * cross(q.v, r), and
      qmul(a, b) = ((b.v * a.w + a.v * b.w) + cross(a.v, b.v),  a.w * b.w - ((a.x b.x + a.y b.y) + a.z b.z)),
      cross(a, b) = (a.y b.z - a.z b.y, a.z b.x - a.x b.z, a.x b.y - a.y b.x);
  box: qc = (-q.v, q.w); ol = qrot(qc, o - p); dl = qrot(qc, d); per axis k = x, y, z: dl_k == 0 -> miss unless |ol_k| <= s_k; else
      enter = ((dl_k > 0 ? -s_k : s_k) - ol_k) / dl_k, leave = ((dl_k > 0 ? s_k : -s_k) - ol_k) / dl_k, tnear/axis updated on enter > tnear
      (strict), tfar on leave < tfar; hit iff tnear <= tfar and tfar >= 0; tnear > 0: t = tnear, normal = qrot(q, sign * e_axis) with
      sign = dl_axis > 0 ? -1 : 1; otherwise t = 0, normal = 0;
  sphere: m = o - c, a = (d.x d.x + d.y d.y) + d.z d.z, b = (m.x d.x + m.y d.y) + m.z d.z, c' = ((m.x m.x + m.y m.y) + m.z m.z) - r r;
      c' <= 0: t = 0, normal = 0; else disc = b b - a c', hit iff disc >= 0, a > 0 and t = (-b - sqrt(disc)) / a >= 0,
      normal = ((o + t d) - c) / r;
  a ray keeps the smallest t in [0, max_t], ties to the smallest collider index (boxes, then spheres), skipping colliders of ignore_body."""
import numpy as np
from nudge_b200 import scenes

f = np.float32
NO_BODY = scenes.NO_BODY


def _cross(ax, ay, az, bx, by, bz):
    return ay * bz - az * by, az * bx - ax * bz, ax * by - ay * bx


def _qrot(vx, vy, vz, w, rx, ry, rz):
    cx, cy, cz = _cross(vx, vy, vz, rx, ry, rz)
    tx, ty, tz = f(2.0) * cx, f(2.0) * cy, f(2.0) * cz
    ux, uy, uz = _cross(vx, vy, vz, tx, ty, tz)
    return (rx + w * tx) + ux, (ry + w * ty) + uy, (rz + w * tz) + uz


def collider_world(body_xf, box_xf, sphere_xf):
    """k_collider_world's world transforms: a TRANSFORM array, boxes first, then spheres (body field = the collider's body)."""
    cx = np.concatenate([box_xf, sphere_xf])
    b = body_xf[cx["body"]]
    ax, ay, az, aw = (b["rotation"][:, k] for k in range(4))
    bx, by, bz, bw = (cx["rotation"][:, k] for k in range(4))
    px, py, pz = _qrot(ax, ay, az, aw, cx["position"][:, 0], cx["position"][:, 1], cx["position"][:, 2])
    px = px + b["position"][:, 0]; py = py + b["position"][:, 1]; pz = pz + b["position"][:, 2]
    ux, uy, uz = _cross(ax, ay, az, bx, by, bz)
    out = np.zeros(len(cx), scenes.TRANSFORM)
    out["position"] = np.stack([px, py, pz], 1)
    out["body"] = cx["body"]
    out["rotation"] = np.stack([(bx * aw + ax * bw) + ux, (by * aw + ay * bw) + uy, (bz * aw + az * bw) + uz,
                                aw * bw - ((ax * bx + ay * by) + az * bz)], 1)
    return out


def _box_hits(o, d, w, size):
    """o, d: [R, 3]; w: world TRANSFORM [K]; size [K, 3].  Returns hit [R, K], t [R, K], normal [3][R, K]."""
    p, q = w["position"], w["rotation"]
    qx, qy, qz, qw = (q[None, :, k] for k in range(4))
    cx, cy, cz = -qx, -qy, -qz
    O = [o[:, k:k + 1] for k in range(3)]
    D = [d[:, k:k + 1] for k in range(3)]
    ol = _qrot(cx, cy, cz, qw, O[0] - p[None, :, 0], O[1] - p[None, :, 1], O[2] - p[None, :, 2])
    dl = _qrot(cx, cy, cz, qw, D[0], D[1], D[2])
    shape = ol[0].shape
    tnear = np.full(shape, -np.inf, f); tfar = np.full(shape, np.inf, f)
    axis = np.full(shape, -1, np.int8); fail = np.zeros(shape, bool)
    for k in range(3):
        s = size[None, :, k]
        zero = dl[k] == 0
        fail |= zero & ~(np.abs(ol[k]) <= s)
        pos = dl[k] > 0
        enter = (np.where(pos, -s, s) - ol[k]) / dl[k]
        leave = (np.where(pos, s, -s) - ol[k]) / dl[k]
        up = ~zero & (enter > tnear)
        tnear = np.where(up, enter, tnear); axis = np.where(up, np.int8(k), axis)
        tfar = np.where(~zero & (leave < tfar), leave, tfar)
    hit = ~fail & (tnear <= tfar) & (tfar >= 0)
    entering = tnear > 0
    t = np.where(entering, tnear, f(0.0))
    d_axis = np.where(axis == 0, dl[0], np.where(axis == 1, dl[1], dl[2]))
    sg = np.where(d_axis > 0, f(-1.0), f(1.0))
    nl = [np.where(axis == k, sg, f(0.0)) for k in range(3)]
    n = _qrot(qx, qy, qz, qw, *nl)
    n = [np.where(entering, c, f(0.0)) for c in n]
    return hit, t, n


def _sphere_hits(o, d, w, radius):
    c = w["position"]
    r = radius[None, :]
    O = [o[:, k:k + 1] for k in range(3)]
    D = [d[:, k:k + 1] for k in range(3)]
    m = [O[k] - c[None, :, k] for k in range(3)]
    a = (D[0] * D[0] + D[1] * D[1]) + D[2] * D[2]
    b = (m[0] * D[0] + m[1] * D[1]) + m[2] * D[2]
    cc = ((m[0] * m[0] + m[1] * m[1]) + m[2] * m[2]) - r * r
    inside = cc <= 0
    disc = b * b - a * cc
    t = (-b - np.sqrt(np.where(disc >= 0, disc, f(0.0)))) / a
    hit = inside | ((disc >= 0) & (a > 0) & (t >= 0))
    t = np.where(inside, f(0.0), t)
    n = [np.where(inside, f(0.0), ((O[k] + t * D[k]) - c[None, :, k]) / r) for k in range(3)]
    return hit, t, n


def raycast(body_xf, box_xf, box_size, box_tags, sphere_xf, sphere_radius, sphere_tags, rays, chunk_elems=1 << 21):
    """body_xf / box_xf / sphere_xf: TRANSFORM arrays; box_size [n, 3]; sphere_radius [m]; rays: RAY array.  Returns a RAY_HIT array."""
    w = collider_world(body_xf, box_xf, sphere_xf)
    nb = len(box_xf)
    wb, ws = w[:nb], w[nb:]
    size = np.asarray(box_size, f).reshape(-1, 3)
    radius = np.asarray(sphere_radius, f).reshape(-1)
    tags = np.concatenate([np.asarray(box_tags, np.uint32), np.asarray(sphere_tags, np.uint32)])
    body = w["body"]
    K = len(w)
    out = np.zeros(len(rays), scenes.RAY_HIT)
    out["t"] = rays["max_t"]
    out["collider"] = NO_BODY; out["body"] = NO_BODY; out["tag"] = NO_BODY
    if K == 0 or len(rays) == 0:
        return out
    step = max(1, chunk_elems // K)
    with np.errstate(all="ignore"):
        for s0 in range(0, len(rays), step):
            r = rays[s0:s0 + step]
            o = np.ascontiguousarray(r["origin"], f); d = np.ascontiguousarray(r["direction"], f)
            parts = [x for x in (_box_hits(o, d, wb, size) if nb else None, _sphere_hits(o, d, ws, radius) if K > nb else None) if x is not None]
            hit = np.concatenate([p[0] for p in parts], 1)
            t = np.concatenate([p[1] for p in parts], 1)
            n = [np.concatenate([p[2][k] for p in parts], 1) for k in range(3)]
            valid = hit & (body[None, :] != r["ignore_body"][:, None]) & (t <= r["max_t"][:, None])
            key = np.where(valid, t, f(np.inf))
            mins = key.min(1)
            j = np.argmax(valid & (key == mins[:, None]), 1)
            anyv = valid.any(1)
            rows = np.nonzero(anyv)[0]
            jj = j[rows]
            o_ = out[s0:s0 + step]
            o_["t"][rows] = t[rows, jj]
            o_["collider"][rows] = jj
            o_["body"][rows] = body[jj]
            o_["tag"][rows] = tags[jj]
            o_["normal"][rows] = np.stack([n[k][rows, jj] for k in range(3)], 1)
            out[s0:s0 + step] = o_
    return out


def _raycast_args(args):
    return raycast(*args)


def raycast_parallel(body_xf, box_xf, box_size, box_tags, sphere_xf, sphere_radius, sphere_tags, rays, workers=None):
    """raycast() with the rays split across worker processes (spawned: safe next to a CUDA context).  Same result, bit for bit."""
    import concurrent.futures as cf
    import multiprocessing as mp
    import os
    workers = max(1, min(workers or os.cpu_count() or 1, 32, len(rays)))
    if workers == 1:
        return raycast(body_xf, box_xf, box_size, box_tags, sphere_xf, sphere_radius, sphere_tags, rays)
    parts = np.array_split(rays, workers)
    with cf.ProcessPoolExecutor(workers, mp_context=mp.get_context("spawn")) as ex:
        out = list(ex.map(_raycast_args, [(body_xf, box_xf, box_size, box_tags, sphere_xf, sphere_radius, sphere_tags, p) for p in parts]))
    return np.concatenate(out)


def raycast_scene(state, rays, parallel=False, **kw):
    """raycast() on anything with the scene arrays (a Scene, a Sim's host state after download_bodies)."""
    fn = raycast_parallel if parallel else raycast
    return fn(state.transforms, state.box_transforms, state.box_data["size"], state.box_tags, state.sphere_transforms,
              state.sphere_data["radius"], state.sphere_tags, rays, **kw)
