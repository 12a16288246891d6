"""nudge_b200 — B200-native rigid-body simulation step, drop-in for rasmusbarr/nudge's hot path.

This package is only the Python binding used by tests and bench.py: it loads the C-ABI shared library
(include/nudge_b200.h, built by nudge_b200/csrc/build.sh) with ctypes and mirrors the reference's seven calls
(nudge.h:134-146) on a device-resident simulation.  There is no CPU path: importing works without a GPU
(so the symbol check can run), creating a `Sim` does not."""
import ctypes as C
import os
import numpy as np
from . import abi, scenes

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libnudge_b200.so")

EXPORTS = ["nb_create", "nb_destroy", "nb_last_error", "nb_upload_bodies", "nb_upload_colliders", "nb_upload_connections", "nb_upload_cache",
           "nb_upload_contacts", "nb_download_bodies", "nb_download_contacts", "nb_download_cache", "nb_download_counts", "nb_upload_momentum", "nb_upload_transforms",
           "nb_download_momentum", "nb_download_transforms", "nb_collide", "nb_apply_gravity_damping", "nb_read_cached_impulses",
           "nb_setup_contact_constraints", "nb_apply_impulses", "nb_update_cached_impulses", "nb_write_cached_impulses", "nb_advance", "nb_step",
           "nb_launch_count", "nb_debug_read", "nb_debug_rcp", "nb_lut_model_exact", "nb_debug_sort", "nb_debug_scan", "nb_debug_enable", "nb_pack_momentum", "nb_unpack_momentum",
           "nb_shard_unique_id", "nb_shard_create", "nb_shard_destroy", "nb_shard_ipc_handle", "nb_shard_open_peer", "nb_shard_plan", "nb_shard_exchange",
           "nb_shard_step", "nb_shard_graph_active", "nb_shard_partition", "nb_shard_debug_no_exchange",
           "nb_set_solver_mode", "nb_get_solver_mode", "nb_debug_timing_enable", "nb_debug_timing",
           "nb_stream_create", "nb_stream_destroy", "nb_stream_synchronize", "nb_save_state", "nb_load_state", "nb_state_info",
           "nb_upload_constraint_rows", "nb_download_constraint_rows", "nb_instance_matrices", "nb_shard_build_plan", "nb_shard_local_scene",
           "nb_build_query_tree", "nb_raycast"]


class Config(C.Structure):
    _fields_ = [("max_bodies", C.c_uint32), ("max_boxes", C.c_uint32), ("max_spheres", C.c_uint32), ("max_connections", C.c_uint32),
                ("max_pairs", C.c_uint32), ("max_contacts", C.c_uint32), ("device", C.c_int)]


class Counts(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in ("pairs", "live_pairs", "contacts", "sleeping", "active", "cache", "culled", "batches", "levels", "overflow")]


_lib = None


def load_library():
    """Loads the CUDA extension; raises if it has not been built (there is no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("nudge_b200: %s is missing — run nudge_b200/csrc/build.sh (or __graft_entry__.build()); there is no CPU path" % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        V = C.c_void_p
        lib.nb_create.argtypes = [V, V]
        lib.nb_destroy.argtypes = [V]
        lib.nb_last_error.argtypes = [V]; lib.nb_last_error.restype = C.c_char_p
        for f in ("nb_upload_bodies", "nb_upload_colliders", "nb_upload_connections", "nb_upload_cache", "nb_download_bodies", "nb_download_cache", "nb_download_counts"):
            getattr(lib, f).argtypes = [V, V, V]
        lib.nb_download_contacts.argtypes = [V, V, V, V]
        lib.nb_upload_contacts.argtypes = [V, V, V, V]
        for f in ("nb_upload_momentum", "nb_upload_transforms", "nb_download_momentum", "nb_download_transforms"):
            getattr(lib, f).argtypes = [V, V, C.c_uint32, V]
        for f in ("nb_collide", "nb_read_cached_impulses", "nb_setup_contact_constraints", "nb_update_cached_impulses", "nb_write_cached_impulses"):
            getattr(lib, f).argtypes = [V, V]
        lib.nb_apply_gravity_damping.argtypes = [V, C.c_float, C.c_float, C.c_float, V]
        lib.nb_apply_impulses.argtypes = [V, C.c_uint32, V]
        lib.nb_advance.argtypes = [V, C.c_float, V]
        lib.nb_step.argtypes = [V, C.c_float, C.c_uint32, C.c_float, C.c_float, V]
        lib.nb_launch_count.argtypes = [V]; lib.nb_launch_count.restype = C.c_uint64
        lib.nb_debug_read.argtypes = [V, C.c_char_p, V, C.c_size_t, V, V]
        lib.nb_debug_rcp.argtypes = [V, V, V, C.c_uint32, C.c_int]
        lib.nb_lut_model_exact.argtypes = [V]
        lib.nb_debug_sort.argtypes = [V, V, V, C.c_uint32, C.c_int, C.c_int]
        lib.nb_debug_scan.argtypes = [V, V, C.c_uint32, V]
        lib.nb_debug_enable.argtypes = [V, C.c_int]
        lib.nb_pack_momentum.argtypes = [V, V, C.c_uint32, V, V]
        lib.nb_unpack_momentum.argtypes = [V, V, V, C.c_uint32, V, V]
        lib.nb_shard_unique_id.argtypes = [V]
        lib.nb_shard_create.argtypes = [V, C.c_uint32, C.c_uint32, V, C.c_uint32, C.c_uint32, V]
        lib.nb_shard_destroy.argtypes = [V]; lib.nb_shard_destroy.restype = None
        lib.nb_shard_ipc_handle.argtypes = [V, V]
        lib.nb_shard_open_peer.argtypes = [V, C.c_uint32, V]
        lib.nb_shard_plan.argtypes = [V, V, C.c_uint32, V, V, V, V, V, C.c_uint32, C.c_uint32, V]
        lib.nb_shard_exchange.argtypes = [V, C.c_int, V]
        lib.nb_shard_step.argtypes = [V, C.c_float, C.c_uint32, C.c_float, C.c_float, C.c_int, V]
        lib.nb_shard_graph_active.argtypes = [V]
        lib.nb_shard_debug_no_exchange.argtypes = [V, C.c_int]
        lib.nb_shard_partition.argtypes = [V, V, C.c_uint32, C.c_uint32, C.c_uint32, C.c_float, C.c_uint32, V, V, V, C.c_uint32]
        lib.nb_set_solver_mode.argtypes = [V, C.c_int]
        lib.nb_get_solver_mode.argtypes = [V]
        lib.nb_debug_timing_enable.argtypes = [V, C.c_int]
        lib.nb_debug_timing.argtypes = [V, V, V, V]
        lib.nb_stream_create.argtypes = [V]; lib.nb_stream_create.restype = V
        lib.nb_stream_destroy.argtypes = [V, V]; lib.nb_stream_destroy.restype = None
        lib.nb_stream_synchronize.argtypes = [V, V]
        lib.nb_save_state.argtypes = [V, C.c_char_p, V]
        lib.nb_load_state.argtypes = [V, C.c_char_p, V]
        lib.nb_state_info.argtypes = [C.c_char_p, V]
        lib.nb_upload_constraint_rows.argtypes = [V, V, C.c_uint32, V]
        lib.nb_download_constraint_rows.argtypes = [V, V, C.c_uint32, V]
        lib.nb_instance_matrices.argtypes = [V, V, C.c_uint32, C.c_int, V, V]
        lib.nb_build_query_tree.argtypes = [V, V]
        lib.nb_raycast.argtypes = [V, V, V, C.c_uint32, C.c_int, V]
        lib.nb_shard_build_plan.argtypes = [V, C.c_uint32, V, V, C.c_uint32, C.c_uint32, V, V, V, V, V, V, V, V]
        lib.nb_shard_local_scene.argtypes = [V, C.c_uint32, V, C.c_uint32, C.c_uint32, V, C.c_uint32, V, C.c_uint32, V, V, V, V, V]
        _lib = lib
    return _lib


class NudgeError(RuntimeError):
    pass


# nb_constraint_row (80 bytes)
ROW = np.dtype([("a", "<u4"), ("b", "<u4"), ("lin_a", "<f4", 3), ("ang_a", "<f4", 3), ("lin_b", "<f4", 3), ("ang_b", "<f4", 3),
                ("bias", "<f4"), ("lo", "<f4"), ("hi", "<f4"), ("impulse", "<f4"), ("softness", "<f4"), ("reserved", "<f4")])
assert ROW.itemsize == 80
# nb_ray / nb_ray_hit (32 bytes each) and the "no body" marker: defined with the other record types in scenes.py
RAY, RAY_HIT, NO_BODY, make_rays = scenes.RAY, scenes.RAY_HIT, scenes.NO_BODY, scenes.make_rays


def nccl_unique_id():
    """128 bytes from ncclGetUniqueId (rank 0 calls it and broadcasts them)."""
    buf = (C.c_ubyte * 128)()
    r = load_library().nb_shard_unique_id(buf)
    if r != 0:
        raise NudgeError("nb_shard_unique_id failed (%d): NCCL not loadable" % r)
    return bytes(buf)


def shard_partition(pos, radius, gx, gz, margin, balance=0):
    """nb_shard_partition (C++ host code, runs without a GPU): owner[n] and the ghost list of every rank."""
    lib = load_library()
    pos = np.ascontiguousarray(pos, np.float32); radius = np.ascontiguousarray(radius, np.float32)
    n, world = len(radius), gx * gz
    owner = np.zeros(n, np.uint32); off = np.zeros(world + 1, np.uint32)
    cap = max(1024, n)
    while True:
        ids = np.zeros(cap, np.uint32)
        r = lib.nb_shard_partition(abi.ptr(pos), abi.ptr(radius), n, int(gx), int(gz), C.c_float(margin), int(balance), abi.ptr(owner), abi.ptr(off), abi.ptr(ids), cap)
        if r == 0:
            break
        if r != -2:
            raise NudgeError("nb_shard_partition failed (%d)" % r)
        cap = int(off[world]) + 16
    return owner, [ids[off[k]:off[k + 1]].copy() for k in range(world)]


def shard_build_plan(owner, ghost_lists, rank):
    """nb_shard_build_plan (C++ host code, runs without a GPU): the exchange plan of `rank` from a partition (owner[n], one 0-based ascending
    ghost id list per rank).  Returns a dict with the arrays nb_shard_plan takes plus owned_ids and max_export."""
    lib = load_library()
    owner = np.ascontiguousarray(owner, np.uint32)
    world = len(ghost_lists)
    off = np.zeros(world + 1, np.uint32)
    off[1:] = np.cumsum([len(g) for g in ghost_lists])
    ids = np.ascontiguousarray(np.concatenate([np.asarray(g, np.uint32) for g in ghost_lists]) if off[world] else np.zeros(1, np.uint32), np.uint32)
    sizes = (C.c_uint32 * 5)()
    r = lib.nb_shard_build_plan(abi.ptr(owner), len(owner), abi.ptr(off), abi.ptr(ids), world, int(rank), sizes, None, None, None, None, None, None, None)
    if r != 0:
        raise NudgeError("nb_shard_build_plan failed (%d)" % r)
    n_owned, n_export, n_ghost, n_sub, max_export = (int(x) for x in sizes)
    A = lambda k: np.zeros(max(int(k), 1), np.uint32)
    owned, exp, so, sr, ss, gl, gs = A(n_owned), A(n_export), A(n_export + 1), A(n_sub), A(n_sub), A(n_ghost), A(n_ghost)
    r = lib.nb_shard_build_plan(abi.ptr(owner), len(owner), abi.ptr(off), abi.ptr(ids), world, int(rank), sizes, abi.ptr(owned), abi.ptr(exp), abi.ptr(so), abi.ptr(sr), abi.ptr(ss), abi.ptr(gl), abi.ptr(gs))
    if r != 0:
        raise NudgeError("nb_shard_build_plan failed (%d)" % r)
    return dict(owned_ids=owned[:n_owned], export_local=exp[:n_export], sub_off=so[:n_export + 1], sub_rank=sr[:n_sub], sub_slot=ss[:n_sub],
                ghost_local=gl[:n_ghost], ghost_src=gs[:n_ghost], max_export=max_export)


def shard_local_scene(owned_ids, ghost_ids, n_bodies_global, box_body, sphere_body):
    """nb_shard_local_scene (C++ host code): (box_sel, box_local_body, sphere_sel, sphere_local_body) for the local scene
    [world body, owned_ids + 1 ..., ghost_ids + 1 ...] (ids 0-based as in shard_partition)."""
    lib = load_library()
    o = np.ascontiguousarray(owned_ids, np.uint32); g = np.ascontiguousarray(ghost_ids, np.uint32)
    bb = np.ascontiguousarray(box_body, np.uint32); sb = np.ascontiguousarray(sphere_body, np.uint32)
    P = lambda a: abi.ptr(a) if len(a) else None
    sizes = (C.c_uint32 * 2)()
    r = lib.nb_shard_local_scene(P(o), len(o), P(g), len(g), int(n_bodies_global), P(bb), len(bb), P(sb), len(sb), sizes, None, None, None, None)
    if r != 0:
        raise NudgeError("nb_shard_local_scene failed (%d)" % r)
    kb, ks = int(sizes[0]), int(sizes[1])
    A = lambda k: np.zeros(max(k, 1), np.uint32)
    bsel, bloc, ssel, sloc = A(kb), A(kb), A(ks), A(ks)
    r = lib.nb_shard_local_scene(P(o), len(o), P(g), len(g), int(n_bodies_global), P(bb), len(bb), P(sb), len(sb), sizes, abi.ptr(bsel), abi.ptr(bloc), abi.ptr(ssel), abi.ptr(sloc))
    if r != 0:
        raise NudgeError("nb_shard_local_scene failed (%d)" % r)
    return bsel[:kb], bloc[:kb], ssel[:ks], sloc[:ks]


class Sim(abi.HostState):
    """Device-resident simulation mirroring the reference's call sequence (example/main.cpp:274-328).

    Host arrays (self.transforms, self.momentum, ...) are the caller-owned copies; `upload()` / `download_bodies()`
    move them across.  `stream` is a raw cudaStream_t (0 = default stream)."""

    def __init__(self, scene, contact_capacity=None, pair_capacity=None, device=0, stream=0, debug=False, max_bodies=None, max_boxes=None, max_spheres=None):
        """max_* reserve room for scenes loaded later with reload() (a sharded scene changes size when it is re-partitioned)."""
        mb, mx, ms = max(scene.n_bodies, max_bodies or 0), max(scene.n_boxes, max_boxes or 0), max(scene.n_spheres, max_spheres or 0)
        super().__init__(scene, contact_capacity or max(1024, 24 * mb))
        self.lib = load_library()
        self.stream = C.c_void_p(stream)
        cfg = Config(mb, mx, ms, max(1, len(scene.connections)),
                     pair_capacity or max(4096, 16 * (mx + ms)), self.cap, device)
        self.ctx = C.c_void_p()
        r = self.lib.nb_create(C.byref(cfg), C.byref(self.ctx))
        if r != 0:
            msg = self.lib.nb_last_error(self.ctx).decode() if self.ctx else "nb_create failed"
            raise NudgeError("nb_create: %s (%d)" % (msg, r))
        if debug:
            self._ck(self.lib.nb_debug_enable(self.ctx, 1), "nb_debug_enable")
        self.upload()

    def close(self):
        if getattr(self, "shard", None):
            self.lib.nb_shard_destroy(self.shard)
            self.shard = None
        if getattr(self, "ctx", None):
            self.lib.nb_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, r, what):
        if r != 0:
            raise NudgeError("%s: %s (%d)" % (what, self.lib.nb_last_error(self.ctx).decode(), r))

    def reload(self, scene):
        """Replaces the scene (bodies and colliders) inside the same device context; the contact cache in HBM is kept (it is keyed by collider tags)."""
        cap = self.cap
        abi.HostState.__init__(self, scene, cap)
        self._ck(self.lib.nb_upload_bodies(self.ctx, C.byref(self.bodies), self.stream), "nb_upload_bodies")
        self._ck(self.lib.nb_upload_colliders(self.ctx, C.byref(self.colliders), self.stream), "nb_upload_colliders")
        self._ck(self.lib.nb_upload_connections(self.ctx, C.byref(self.conn), self.stream), "nb_upload_connections")

    def pack_momentum(self, dev_indices_ptr, n, dev_out_ptr):
        self._ck(self.lib.nb_pack_momentum(self.ctx, C.c_void_p(dev_indices_ptr), int(n), C.c_void_p(dev_out_ptr), self.stream), "nb_pack_momentum")

    def unpack_momentum(self, dev_indices_ptr, dev_sources_ptr, n, dev_in_ptr):
        self._ck(self.lib.nb_unpack_momentum(self.ctx, C.c_void_p(dev_indices_ptr), C.c_void_p(dev_sources_ptr), int(n), C.c_void_p(dev_in_ptr), self.stream), "nb_unpack_momentum")

    # ---- one scene sharded across GPUs: the C++ host behind nb_shard_* (include/nudge_b200.h) ----
    TRANSPORT = {"nccl": 0, "peer": 1}

    def shard_create(self, rank, world, nccl_id, ghost_capacity, export_capacity):
        self.shard = C.c_void_p()
        idbuf = (C.c_ubyte * 128).from_buffer_copy(nccl_id) if nccl_id is not None else None
        self._ck(self.lib.nb_shard_create(self.ctx, int(rank), int(world), idbuf, int(ghost_capacity), int(export_capacity), C.byref(self.shard)), "nb_shard_create")

    def shard_ipc_handle(self):
        h = (C.c_ubyte * 64)()
        self._ck(self.lib.nb_shard_ipc_handle(self.shard, h), "nb_shard_ipc_handle")
        return bytes(h)

    def shard_open_peer(self, peer, handle):
        self._ck(self.lib.nb_shard_open_peer(self.shard, int(peer), (C.c_ubyte * 64).from_buffer_copy(handle)), "nb_shard_open_peer")

    def shard_plan(self, export_local, sub_off, sub_rank, sub_slot, ghost_local, ghost_src, max_export):
        arrs = [np.ascontiguousarray(x, np.uint32) for x in (export_local, sub_off, sub_rank, sub_slot, ghost_local, ghost_src)]
        e, so, sr, ss, gl, gs = arrs
        self._ck(self.lib.nb_shard_plan(self.shard, abi.ptr(e), len(e), abi.ptr(so), abi.ptr(sr), abi.ptr(ss), abi.ptr(gl), abi.ptr(gs), len(gl), int(max_export), self.stream), "nb_shard_plan")

    def shard_exchange(self, transport):
        self._ck(self.lib.nb_shard_exchange(self.shard, self.TRANSPORT[transport], self.stream), "nb_shard_exchange")

    def shard_step(self, transport):
        s = self.scene
        self._ck(self.lib.nb_shard_step(self.shard, float(s.time_step), int(s.iterations), float(s.gravity), float(s.damping), self.TRANSPORT[transport], self.stream), "nb_shard_step")

    def shard_no_exchange(self, on):
        self._ck(self.lib.nb_shard_debug_no_exchange(self.shard, 1 if on else 0), "nb_shard_debug_no_exchange")

    def shard_graph_active(self):
        return bool(self.lib.nb_shard_graph_active(self.shard))

    # ---- host <-> HBM ----
    def upload(self):
        self._ck(self.lib.nb_upload_bodies(self.ctx, C.byref(self.bodies), self.stream), "nb_upload_bodies")
        self._ck(self.lib.nb_upload_colliders(self.ctx, C.byref(self.colliders), self.stream), "nb_upload_colliders")
        self._ck(self.lib.nb_upload_connections(self.ctx, C.byref(self.conn), self.stream), "nb_upload_connections")
        self._ck(self.lib.nb_upload_cache(self.ctx, C.byref(self.cache), self.stream), "nb_upload_cache")

    def upload_bodies(self):
        self._ck(self.lib.nb_upload_bodies(self.ctx, C.byref(self.bodies), self.stream), "nb_upload_bodies")

    def upload_cache(self):
        self._ck(self.lib.nb_upload_cache(self.ctx, C.byref(self.cache), self.stream), "nb_upload_cache")

    def download_bodies(self):
        self._ck(self.lib.nb_download_bodies(self.ctx, C.byref(self.bodies), self.stream), "nb_download_bodies")

    def download_contacts(self):
        self.contacts.capacity = self.cap
        self.active.capacity = self.scene.n_bodies
        self._ck(self.lib.nb_download_contacts(self.ctx, C.byref(self.contacts), C.byref(self.active), self.stream), "nb_download_contacts")

    def download_cache(self):
        self.cache.capacity = self.cap
        self._ck(self.lib.nb_download_cache(self.ctx, C.byref(self.cache), self.stream), "nb_download_cache")

    def counts(self):
        c = Counts()
        r = self.lib.nb_download_counts(self.ctx, C.byref(c), self.stream)
        if r != -4:   # NB_ERR_OVERFLOW still fills the struct: the caller reads c.overflow
            self._ck(r, "nb_download_counts")
        return c

    # ---- the seven calls + the user loop ----
    def collide(self):
        self._ck(self.lib.nb_collide(self.ctx, self.stream), "nb_collide")

    def apply_gravity_damping(self):
        s = self.scene
        self._ck(self.lib.nb_apply_gravity_damping(self.ctx, float(s.time_step), float(s.gravity), float(s.damping), self.stream), "nb_apply_gravity_damping")

    def read_cached_impulses(self):
        self._ck(self.lib.nb_read_cached_impulses(self.ctx, self.stream), "nb_read_cached_impulses")

    def setup_contact_constraints(self):
        self._ck(self.lib.nb_setup_contact_constraints(self.ctx, self.stream), "nb_setup_contact_constraints")

    def apply_impulses(self, sweeps=1):
        self._ck(self.lib.nb_apply_impulses(self.ctx, int(sweeps), self.stream), "nb_apply_impulses")

    def update_cached_impulses(self):
        self._ck(self.lib.nb_update_cached_impulses(self.ctx, self.stream), "nb_update_cached_impulses")

    def write_cached_impulses(self):
        self._ck(self.lib.nb_write_cached_impulses(self.ctx, self.stream), "nb_write_cached_impulses")

    def advance(self):
        self._ck(self.lib.nb_advance(self.ctx, float(self.scene.time_step), self.stream), "nb_advance")

    def step(self):
        s = self.scene
        self._ck(self.lib.nb_step(self.ctx, float(s.time_step), int(s.iterations), float(s.gravity), float(s.damping), self.stream), "nb_step")

    def step_staged(self):
        """The same sub-step through the seven stage calls (example/main.cpp:274-328)."""
        self.collide(); self.apply_gravity_damping(); self.read_cached_impulses(); self.setup_contact_constraints()
        self.apply_impulses(int(self.scene.iterations)); self.update_cached_impulses(); self.write_cached_impulses(); self.advance()

    def launch_count(self):
        return int(self.lib.nb_launch_count(self.ctx))

    # ---- user constraint rows (nb_constraint_row, include/nudge_b200.h) ----
    def upload_constraint_rows(self, rows):
        rows = np.ascontiguousarray(rows, ROW)
        self._ck(self.lib.nb_upload_constraint_rows(self.ctx, abi.ptr(rows) if len(rows) else None, len(rows), self.stream), "nb_upload_constraint_rows")

    def download_constraint_rows(self, n):
        rows = np.zeros(n, ROW)
        self._ck(self.lib.nb_download_constraint_rows(self.ctx, abi.ptr(rows) if n else None, n, self.stream), "nb_download_constraint_rows")
        return rows

    # ---- renderer read-back (example/main.cpp:224-268): one column-major 4x4 model matrix per collider, boxes first, then spheres ----
    def instance_matrices(self, out=None, device_ptr=None, capacity=0):
        """Host destination (default): returns an (n, 16) float32 array.  device_ptr: writes into that device buffer (e.g. a mapped
        graphics resource) asynchronously on the Sim's stream and returns the collider count."""
        n = C.c_uint32(0)
        if device_ptr is not None:
            self._ck(self.lib.nb_instance_matrices(self.ctx, C.c_void_p(device_ptr), capacity, 1, C.byref(n), self.stream), "nb_instance_matrices")
            return int(n.value)
        k = self.scene.n_colliders
        if out is None:
            out = np.zeros((k, 16), np.float32)
        self._ck(self.lib.nb_instance_matrices(self.ctx, abi.ptr(out), len(out), 0, C.byref(n), self.stream), "nb_instance_matrices")
        return out[:n.value]

    # ---- ray casts against a snapshot of the scene (nb_build_query_tree / nb_raycast, include/nudge_b200.h) ----
    def build_query_tree(self):
        """Snapshots the scene as it is now (transforms, colliders, sizes, tags) and builds the query tree; asynchronous on the Sim's stream."""
        self._ck(self.lib.nb_build_query_tree(self.ctx, self.stream), "nb_build_query_tree")

    def raycast(self, origins=None, directions=None, max_t=np.inf, ignore_body=None, rays=None, device_ptr=None, hits_ptr=None, n=0):
        """Casts rays against the last snapshot.  Host form: origins / directions [n, 3] (or a RAY array as `rays`), max_t and ignore_body
        scalars or [n] arrays; returns a RAY_HIT array.  Device form: device_ptr = device address of n RAY records, hits_ptr = device
        address for n RAY_HIT records (e.g. torch tensors' data_ptr()); asynchronous on the Sim's stream, returns None."""
        if device_ptr is not None:
            self._ck(self.lib.nb_raycast(self.ctx, C.c_void_p(device_ptr), C.c_void_p(hits_ptr), int(n), 1, self.stream), "nb_raycast")
            return None
        r = np.ascontiguousarray(rays if rays is not None else scenes.make_rays(origins, directions, max_t, ignore_body), scenes.RAY)
        hits = np.zeros(len(r), scenes.RAY_HIT)
        self._ck(self.lib.nb_raycast(self.ctx, abi.ptr(r) if len(r) else None, abi.ptr(hits) if len(r) else None, len(r), 0, self.stream), "nb_raycast")
        return hits

    # ---- state files (nb_save_state / nb_load_state; tools/nb_replay steps them headless) ----
    def save_state(self, path):
        self._ck(self.lib.nb_save_state(self.ctx, os.fsencode(path), self.stream), "nb_save_state")

    def load_state(self, path):
        self._ck(self.lib.nb_load_state(self.ctx, os.fsencode(path), self.stream), "nb_load_state")

    # ---- solver mode (include/nudge_b200.h): "parity" = the reference's exact Gauss-Seidel order, "throughput" = mass-splitting Jacobi ----
    def set_solver_mode(self, mode):
        self._ck(self.lib.nb_set_solver_mode(self.ctx, {"parity": 0, "throughput": 1}[mode]), "nb_set_solver_mode")

    def solver_mode(self):
        return ["parity", "throughput"][int(self.lib.nb_get_solver_mode(self.ctx))]

    def timing_enable(self, on=True):
        self._ck(self.lib.nb_debug_timing_enable(self.ctx, 1 if on else 0), "nb_debug_timing_enable")

    def timing(self):
        """(launches, total milliseconds) of the dominant solver kernel since the last call (CUDA events inside the library)."""
        n = C.c_uint32(0); ms = C.c_float(0.0)
        self._ck(self.lib.nb_debug_timing(self.ctx, C.byref(n), C.byref(ms), self.stream), "nb_debug_timing")
        return int(n.value), float(ms.value)

    def lut_model_exact(self):
        return bool(self.lib.nb_lut_model_exact(self.ctx))

    # ---- parity-test introspection ----
    def debug(self, name, dtype):
        n = C.c_size_t(0)
        self._ck(self.lib.nb_debug_read(self.ctx, name.encode(), None, 0, C.byref(n), self.stream), "nb_debug_read")
        buf = np.zeros(max(n.value, 1), np.uint8)
        if n.value:
            self._ck(self.lib.nb_debug_read(self.ctx, name.encode(), abi.ptr(buf), n.value, C.byref(n), self.stream), "nb_debug_read")
        return buf[:n.value].view(dtype)

    def debug_scalar(self, name):
        v = np.zeros(1, np.uint32); n = C.c_size_t(0)
        self._ck(self.lib.nb_debug_read(self.ctx, name.encode(), abi.ptr(v), 4, C.byref(n), self.stream), "nb_debug_read")
        return int(v[0])

    def device_rcp(self, x, rsqrt=False):
        x = np.ascontiguousarray(x, np.float32); y = np.empty_like(x)
        for b in range(0, len(x), 1024):
            xs = np.ascontiguousarray(x[b:b + 1024]); ys = np.empty_like(xs)
            self._ck(self.lib.nb_debug_rcp(self.ctx, abi.ptr(xs), abi.ptr(ys), len(xs), 1 if rsqrt else 0), "nb_debug_rcp")
            y[b:b + 1024] = ys
        return y

    def device_sort(self, keys, vals=None, begin_bit=0, end_bit=64):
        keys = np.ascontiguousarray(keys, np.uint64).copy()
        v = np.ascontiguousarray(vals, np.uint32).copy() if vals is not None else None
        self._ck(self.lib.nb_debug_sort(self.ctx, abi.ptr(keys), abi.ptr(v) if v is not None else None, len(keys), begin_bit, end_bit), "nb_debug_sort")
        return keys, v

    def device_scan(self, data):
        d = np.ascontiguousarray(data, np.uint32).copy(); total = np.zeros(1, np.uint32)
        self._ck(self.lib.nb_debug_scan(self.ctx, abi.ptr(d), len(d), abi.ptr(total)), "nb_debug_scan")
        return d, int(total[0])

    def pairs_view(self):
        kbits = self.debug_scalar("kbits")
        keys = self.debug("pair_keys", np.uint64)
        return dict(lo=(keys & np.uint64((1 << kbits) - 1)).astype(np.uint32), hi=(keys >> np.uint64(kbits)).astype(np.uint32), order=self.debug("order", np.uint32))

    def impulses_view(self):
        return dict(sorted=self.debug("sorted", np.uint32), data=self.debug("impulses", scenes.IMPULSE),
                    culled_tags=self.debug("culled_tags", np.uint64), culled_features=self.debug("culled_features", np.uint32),
                    culled_data=self.debug("culled_data", scenes.IMPULSE))

    def constraints_view(self):
        """Rows and states per occupied slot (slot = batch*8 + lane, the reference's ContactConstraintV lane), keyed by contact index."""
        stride = self.debug_scalar("row_stride")
        slot_contact = self.debug("row_contact", np.uint32)
        used = np.nonzero(slot_contact != 0xffffffff)[0]
        planes = self.debug("row_planes", np.float32).reshape(39, stride)[:, used]
        states = self.debug("row_states", np.float32).reshape(3, stride)[:, used]
        sorted_c = self.debug("sorted", np.uint32)
        n = len(sorted_c)
        batch = np.zeros(n, np.uint32); batch[sorted_c] = self.debug("batch_of", np.uint32)
        slot = np.zeros(n, np.uint32); slot[sorted_c] = self.debug("slot_idx", np.uint32)
        return dict(contact=slot_contact[used], a=self.debug("row_a", np.uint32)[used], b=self.debug("row_b", np.uint32)[used], rows=planes.T.copy(), states=states.T.copy(),
                    batch_of_contact=batch, slot_of_contact=slot, slots=used.astype(np.uint32))
