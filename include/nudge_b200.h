/* nudge_b200 — C ABI of the B200-native rigid-body simulation step (drop-in for rasmusbarr/nudge's hot path).
 *
 * Every entry point replaces one reference interface (file:line into /root/reference):
 *
 *   nb_collide                      <- nudge::collide                    nudge.h:134, nudge.cpp:3000-4009
 *   nb_read_cached_impulses         <- nudge::read_cached_impulses       nudge.h:136, nudge.cpp:4021-4108
 *   nb_write_cached_impulses        <- nudge::write_cached_impulses      nudge.h:138, nudge.cpp:4110-4158
 *   nb_setup_contact_constraints    <- nudge::setup_contact_constraints  nudge.h:140, nudge.cpp:4170-4638
 *   nb_apply_impulses               <- nudge::apply_impulses             nudge.h:142, nudge.cpp:4640-4855
 *   nb_update_cached_impulses       <- nudge::update_cached_impulses     nudge.h:144, nudge.cpp:4857-4884
 *   nb_advance                      <- nudge::advance                    nudge.h:146, nudge.cpp:4886-4926
 *   nb_apply_gravity_damping        <- the user loop of example/main.cpp:291-305
 *   nb_step                         <- simulate(), example/main.cpp:274-328 (one sub-step)
 *   nb_upload_connections           <- BodyConnections of nudge::collide  nudge.h:108-111, example/main.cpp:285
 *   nb_upload_contacts              <- "custom contacts can be added here" example/main.cpp:288
 *   nb_upload_constraint_rows       <- "custom constraint impulses"        example/main.cpp:316
 *   nb_instance_matrices            <- the draw loops of render()          example/main.cpp:224-268 (helpers :53-110)
 *   nb_save_state / nb_load_state   <- the caller-owned PODs               nudge.h:73-129
 *   nb_shard_*                      <- no reference counterpart (the reference is single threaded): SURVEY.md section 8e
 *   nb_build_query_tree, nb_raycast <- no reference counterpart (ray queries): DESIGN.md section 8.5
 *
 * Data layout: the reference's caller-owned SoA structs (nudge.h:29-129) with every index-carrying field
 * widened to 32 bits (the reference caps at 8192 colliders / 65535 bodies, nudge.cpp:3010, nudge.h:68-71):
 *
 *   BodyPair{uint16 a,b}                             -> nb_body_pair{uint32 a,b}
 *   collider tag uint16                              -> uint32
 *   contact tag uint64 = feature | A<<32 | B<<48     -> tags[i] = A | (uint64)B<<32 ; features[i] = feature
 *   sleeping pair uint32 = X | Y<<16                 -> uint64 = X | (uint64)Y<<32
 *   ActiveBodies.indices uint16                      -> uint32
 *
 * The simulation state is DEVICE RESIDENT inside an nb_context (HBM); nb_upload_* / nb_download_* move the
 * caller's host arrays across.  All calls are asynchronous on the given CUDA stream unless stated; no call
 * falls back to the CPU — if the GPU or the CUDA extension is missing, nb_create fails.
 * The uint16 drop-in with the exact nudge.h signatures lives in nudge_b200/csrc/nudge_compat.cpp.
 *
 * Return value: 0 on success, otherwise a negative nb_status; nb_last_error() gives the text.
 */
#ifndef NUDGE_B200_H
#define NUDGE_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct { float position[3]; uint32_t body; float rotation[4]; } nb_transform;          /* nudge.h:34-38 */
typedef struct { float inertia_inverse[3]; float mass_inverse; } nb_body_properties;            /* nudge.h:40-43 */
typedef struct { float velocity[3]; float unused0; float angular_velocity[3]; float unused1; } nb_body_momentum; /* nudge.h:45-50 */
typedef struct { float radius; } nb_sphere_collider;                                            /* nudge.h:52-54 */
typedef struct { float size[3]; float unused; } nb_box_collider;                                /* nudge.h:56-59 */
typedef struct { float position[3]; float penetration; float normal[3]; float friction; } nb_contact; /* nudge.h:61-66 */
typedef struct { uint32_t a, b; } nb_body_pair;                                                 /* nudge.h:68-71, widened */
typedef struct { float impulse[3]; float unused; } nb_cached_impulse;                           /* nudge.h:109-112 */

typedef struct {                                                                                /* nudge.h:73-82 */
	nb_contact* data; nb_body_pair* bodies; uint64_t* tags; uint32_t* features;
	uint32_t capacity, count;
	uint64_t* sleeping_pairs; uint32_t sleeping_count;
} nb_contact_data;

typedef struct { uint32_t* tags; nb_box_collider* data; nb_transform* transforms; uint32_t count; } nb_box_colliders;
typedef struct { uint32_t* tags; nb_sphere_collider* data; nb_transform* transforms; uint32_t count; } nb_sphere_colliders;
typedef struct { nb_box_colliders boxes; nb_sphere_colliders spheres; } nb_collider_data;        /* nudge.h:84-98 */
typedef struct { nb_transform* transforms; nb_body_properties* properties; nb_body_momentum* momentum; uint8_t* idle_counters; uint32_t count; } nb_body_data; /* nudge.h:100-106 */
typedef struct { nb_body_pair* data; uint32_t count; } nb_body_connections;                      /* nudge.h:108-111 */
typedef struct { uint64_t* tags; uint32_t* features; nb_cached_impulse* data; uint32_t capacity, count; } nb_contact_cache; /* nudge.h:114-119 */
typedef struct { uint32_t* indices; uint32_t capacity, count; } nb_active_bodies;                /* nudge.h:121-125 */

typedef struct nb_context nb_context;

typedef struct {
	uint32_t max_bodies, max_boxes, max_spheres, max_connections;
	uint32_t max_pairs;     /* broadphase pairs (about 7 per collider in a pile); 0 = 16 per collider */
	uint32_t max_contacts;  /* also the contact-cache capacity; 0 = 24 per body */
	int device;             /* CUDA device ordinal */
} nb_config;

enum nb_status { NB_OK = 0, NB_ERR_CUDA = -1, NB_ERR_CAPACITY = -2, NB_ERR_ARGUMENT = -3, NB_ERR_OVERFLOW = -4 };

/* Device counters of the last step (copied by nb_download_counts; synchronises the stream). */
typedef struct {
	uint32_t pairs, live_pairs, contacts, sleeping, active, cache, culled, batches, levels, overflow;
} nb_counts;

int nb_create(const nb_config* config, nb_context** out);
void nb_destroy(nb_context* ctx);
const char* nb_last_error(const nb_context* ctx);

/* Host <-> HBM.  Counts in the structs say how many rows to move; pointers are HOST pointers. */
/* nb_upload_bodies is asynchronous (keep the host arrays unchanged until the next synchronising call; pin them to get real overlap): on a created
 * stream the momentum and property rows travel on the library's own copy stream while `stream` goes on with the collision stage, and whatever
 * reads them first on `stream` is ordered after the copy by the library (NB_COPY_OVERLAP=0 disables it).  Use ONE stream per context. */
int nb_upload_bodies(nb_context*, const nb_body_data* host, void* stream);
int nb_upload_colliders(nb_context*, const nb_collider_data* host, void* stream);
int nb_upload_connections(nb_context*, const nb_body_connections* host, void* stream);
int nb_upload_cache(nb_context*, const nb_contact_cache* host, void* stream);
int nb_upload_contacts(nb_context*, const nb_contact_data* host /* may be null */, const nb_active_bodies* host_active /* may be null */, void* stream); /* synchronises */
int nb_download_bodies(nb_context*, nb_body_data* host, void* stream);
int nb_download_contacts(nb_context*, nb_contact_data* host, nb_active_bodies* host_active, void* stream); /* synchronises */
int nb_download_cache(nb_context*, nb_contact_cache* host, void* stream);                                  /* synchronises */
int nb_download_counts(nb_context*, nb_counts* out, void* stream);   /* synchronises; fills *out and returns NB_ERR_OVERFLOW when out->overflow != 0 */
int nb_upload_momentum(nb_context*, const nb_body_momentum* host, uint32_t count, void* stream);
int nb_upload_transforms(nb_context*, const nb_transform* host, uint32_t count, void* stream);
int nb_download_momentum(nb_context*, nb_body_momentum* host, uint32_t count, void* stream);
int nb_download_transforms(nb_context*, nb_transform* host, uint32_t count, void* stream);

/* Ghost exchange of a scene sharded across GPUs: gather momentum rows of `dev_indices` into a contiguous DEVICE buffer (n x 32 B), and
 * scatter rows `dev_sources[i]` of a DEVICE buffer into body `dev_indices[i]`.  The buffer in between travels through one ncclAllGather. */
int nb_pack_momentum(nb_context*, const uint32_t* dev_indices, uint32_t n, void* dev_out, void* stream);
int nb_unpack_momentum(nb_context*, const uint32_t* dev_indices, const uint32_t* dev_sources, uint32_t n, const void* dev_in, void* stream);

/* One scene sharded across GPUs (SURVEY.md section 8e): C++ host, one process or thread per GPU, one nb_context per rank holding the
 * rank's OWNED bodies plus GHOST copies of neighbouring bodies.  After the warm start and after every solver sweep the ghosts'
 * BodyMomentum rows are replaced by their owners' (nb_shard_exchange), either with ONE ncclAllGather (NB_SHARD_NCCL, what BASELINE.json
 * prescribes; NCCL is bound at run time with dlopen) or with this library's own push/pull kernels over CUDA-IPC peer memory
 * (NB_SHARD_PEER: neighbour-only traffic over NVLink, no collective).  Both give bit-identical ghost rows.
 *   rank 0: nb_shard_unique_id -> broadcast the 128 bytes -> every rank: nb_shard_create;  every rank: nb_shard_ipc_handle -> all-gather
 *   the 64-byte handles -> nb_shard_open_peer for every other rank;  after every (re)partition: nb_shard_plan;  then nb_shard_step per
 *   sub-step (or nb_shard_exchange between the stage calls).  nb_shard_partition is the (host, deterministic) partition rule. */
typedef struct nb_shard nb_shard;
enum nb_shard_transport { NB_SHARD_NCCL = 0, NB_SHARD_PEER = 1 };
int nb_shard_unique_id(void* nccl_id_out /* 128 bytes */);
int nb_shard_create(nb_context*, uint32_t rank, uint32_t world, const void* nccl_id /* null: peer transport only */, uint32_t ghost_capacity, uint32_t export_capacity, nb_shard** out);
void nb_shard_destroy(nb_shard*);
int nb_shard_ipc_handle(nb_shard*, void* handle_out /* 64 bytes */);
int nb_shard_open_peer(nb_shard*, uint32_t peer, const void* handle);
int nb_shard_plan(nb_shard*, const uint32_t* export_local, uint32_t n_export, const uint32_t* sub_off, const uint32_t* sub_rank, const uint32_t* sub_slot,
                  const uint32_t* ghost_local, const uint32_t* ghost_src, uint32_t n_ghost, uint32_t max_export, void* stream);
int nb_shard_exchange(nb_shard*, int transport, void* stream);
int nb_shard_step(nb_shard*, float time_step, uint32_t iterations, float gravity, float damping, int transport, void* stream);
int nb_shard_graph_active(const nb_shard*);
int nb_shard_debug_no_exchange(nb_shard*, int on);   /* diagnostic: nb_shard_step runs the rank's local problem without the ghost hand-over */
int nb_shard_partition(const float* pos_xyz, const float* radius, uint32_t n, uint32_t gx, uint32_t gz, float margin, uint32_t balance_iterations,
                       uint32_t* owner_out, uint32_t* ghost_off /* gx*gz + 1 */, uint32_t* ghost_ids, uint32_t ghost_capacity);
/* One rank's exchange plan (the arrays nb_shard_plan takes) from that partition; host code, two passes: with any output null only
 * sizes[] = { n_owned, n_export, n_ghost, n_subscriptions, max_export } is filled.  owned_ids = this rank's bodies (0-based, ascending):
 * local body 1 + k is owned_ids[k], local body 1 + n_owned + j is the j-th entry of the rank's ghost list. */
int nb_shard_build_plan(const uint32_t* owner, uint32_t n, const uint32_t* ghost_off, const uint32_t* ghost_ids, uint32_t world, uint32_t rank,
                        uint32_t sizes[5], uint32_t* owned_ids, uint32_t* export_local, uint32_t* sub_off /* n_export + 1 */, uint32_t* sub_rank, uint32_t* sub_slot,
                        uint32_t* ghost_local, uint32_t* ghost_src);
/* The colliders of one rank's local scene ([world body, owned..., ghosts...]) in the global collider order and the local index of their
 * bodies; host code, two passes (sizes = { kept boxes, kept spheres }). */
int nb_shard_local_scene(const uint32_t* owned_ids, uint32_t n_owned, const uint32_t* ghost_ids, uint32_t n_ghost, uint32_t n_bodies_global,
                         const uint32_t* box_body, uint32_t n_boxes, const uint32_t* sphere_body, uint32_t n_spheres, uint32_t sizes[2],
                         uint32_t* box_sel, uint32_t* box_local_body, uint32_t* sphere_sel, uint32_t* sphere_local_body);

/* The simulation step, device resident.  Same order of calls as example/main.cpp:274-328. */
int nb_collide(nb_context*, void* stream);
int nb_apply_gravity_damping(nb_context*, float time_step, float gravity, float damping, void* stream);
int nb_read_cached_impulses(nb_context*, void* stream);
int nb_setup_contact_constraints(nb_context*, void* stream);
int nb_apply_impulses(nb_context*, uint32_t sweeps, void* stream);  /* `sweeps` back-to-back calls of nudge::apply_impulses */
int nb_update_cached_impulses(nb_context*, void* stream);
int nb_write_cached_impulses(nb_context*, void* stream);
int nb_advance(nb_context*, float time_step, void* stream);
/* One sub-step = the eight calls above in order.  On a stream the caller created (not the legacy default stream) the launches
 * are recorded once into a CUDA graph and replayed; NB_GRAPH=0 in the environment keeps plain launches. */
int nb_step(nb_context*, float time_step, uint32_t iterations, float gravity, float damping, void* stream);

/* User constraint rows (SURVEY.md section 8 f1): the device-resident form of the hook at example/main.cpp:316 ("Custom constraint impulses
 * should be applied here", after every apply_impulses sweep).  One row = one scalar velocity constraint between bodies a and b
 * (0 = the static world):  J v + bias -> 0  with the accumulated impulse kept inside [lo, hi]; rows are applied by sequential impulses in
 * upload order after every contact sweep, their accumulated impulses warm-start the next step (nudge_b200/csrc/nb_rows_api.cuh).
 * Connect the bodies of a joint with nb_upload_connections too, so that islands treat them as one (example/main.cpp:285). */
typedef struct {
	uint32_t a, b;
	float lin_a[3], ang_a[3];   /* Jacobian of body a: linear and angular part */
	float lin_b[3], ang_b[3];   /* Jacobian of body b */
	float bias;                 /* velocity target term (e.g. Baumgarte: beta / dt * position error) */
	float lo, hi;               /* bounds of the accumulated impulse: (-inf, inf) joint, [0, inf) unilateral, [-f, f] motor / friction */
	float impulse;              /* accumulated impulse: warm start on upload, result on download */
	float softness;             /* constraint force mixing added to the effective inverse mass; 0 = rigid */
	float reserved;
} nb_constraint_row;            /* 80 bytes */
int nb_upload_constraint_rows(nb_context*, const nb_constraint_row* host_rows, uint32_t n, void* stream);   /* replaces the set; n = 0 removes it; synchronises */
int nb_download_constraint_rows(nb_context*, nb_constraint_row* host_rows, uint32_t n, void* stream);       /* caller's order; synchronises */

/* CUDA streams for hosts that do not link the CUDA runtime (cgo / JNI / ctypes callers): a created stream is capturable, so nb_step
 * replays its CUDA graph there; a null stream means the legacy default stream and plain launches. */
void* nb_stream_create(nb_context*);
void nb_stream_destroy(nb_context*, void* stream);
int nb_stream_synchronize(nb_context*, void* stream);

/* State serialisation (SURVEY.md section 8 f3): the caller-owned PODs of nudge.h:73-129 (BodyData, ColliderData, BodyConnections,
 * ContactCache, widened layout) as one flat file, from / into the device-resident context.  Checkpoint, and what tools/nb_replay
 * steps headless; layout in nudge_b200/csrc/nb_state_api.cuh.  All three synchronise. */
int nb_save_state(nb_context*, const char* path, void* stream);
int nb_load_state(nb_context*, const char* path, void* stream);
int nb_state_info(const char* path, uint32_t counts[5] /* bodies, boxes, spheres, connections, cache entries */);

/* Renderer read-back (SURVEY.md section 8 f4; replaces the per-collider host loop of example/main.cpp:224-268 with its helpers at :53-110):
 * one column-major 4x4 model matrix (16 floats) per collider, boxes first, then spheres; rotation = body * collider, translation =
 * body.rotation applied to collider.position plus body.position, columns scaled by the box half extents / the sphere radius.
 * out_is_device != 0: `out` is a device pointer (a mapped GL / Vulkan buffer), the call is asynchronous on `stream`; otherwise `out`
 * is host memory and the call returns when it is filled.  *count = colliders; NB_ERR_CAPACITY if capacity (in matrices) is smaller. */
int nb_instance_matrices(nb_context*, float* out, uint32_t capacity, int out_is_device, uint32_t* count, void* stream);

/* Ray casts against the device-resident scene (no reference counterpart; nudge_b200/csrc/nb_query_api.cuh, DESIGN.md section 8.5).
 *
 * nb_build_query_tree takes a SNAPSHOT of the scene as it is now (body transforms, collider transforms, sizes and tags) into buffers of
 * its own, allocated on the first call, and builds an 8-ary AABB tree over it; it never touches what the step uses.  nb_raycast queries
 * the last snapshot, so one build serves any number of ray batches, and rays do not see later nb_advance / nb_step calls until the next
 * build.  io_is_device != 0: rays and hits are device pointers, the call is asynchronous on `stream` and can be captured into the
 * caller's own CUDA graph; otherwise they are host pointers, staged through the library's buffers, and the call synchronises.
 * nb_raycast returns NB_ERR_ARGUMENT when no snapshot exists, when the collider counts changed since it was taken (nb_upload_colliders,
 * nb_load_state), or when a pointer is null while n > 0.
 *
 * Semantics (float32, exact: the same scene and rays give the same bits whatever the tree shape, ray order or launch configuration):
 *  - The hit is the smallest t in [0, max_t] at which origin + t*direction meets a solid collider.  direction need not be unit length;
 *    t is measured in units of it.  origin and direction must be finite.
 *  - Equal t goes to the smallest collider index: boxes 0..nboxes-1, then spheres from nboxes on (the order of nb_instance_matrices).
 *  - Colliders of body ignore_body are skipped; NB_NO_BODY skips nothing.  Body 0 (the static world) is hit like any other body.
 *  - An origin inside a collider (boundary included) gives t = 0 and normal = (0,0,0).
 *  - A miss gives t = max_t, collider = body = tag = NB_NO_BODY and normal = (0,0,0).
 *  - Collider world transform = body * collider, the operations of the collision stage.
 *  - Box: the ray is moved into the box frame (origin - position and direction rotated by the conjugate rotation), then slabs against
 *    the half extents with IEEE division.  A zero direction component makes that axis "inside iff |origin| <= size".  The normal is the
 *    local axis of the entering slab, signed against the direction and rotated to world space; tied slabs go to the lowest axis (x, y, z).
 *  - Sphere: m = origin - centre, a = d.d, b = m.d, c = m.m - r*r, disc = b*b - a*c; inside iff c <= 0; otherwise a hit needs disc >= 0,
 *    a > 0 and t = (-b - sqrt(disc)) / a >= 0, with normal = (origin + t*d - centre) / r.
 *  The exact order of every float operation is fixed in DESIGN.md section 8.5. */
typedef struct { float origin[3]; float max_t; float direction[3]; uint32_t ignore_body; } nb_ray;                        /* 32 B */
typedef struct { float t; uint32_t collider, body, tag; float normal[3]; float unused; } nb_ray_hit;                    /* 32 B */
#define NB_NO_BODY 0xffffffffu   /* ignore_body: skip nothing.  Also collider / body / tag of a miss */
int nb_build_query_tree(nb_context*, void* stream);
int nb_raycast(nb_context*, const nb_ray* rays, nb_ray_hit* hits, uint32_t n, int io_is_device, void* stream);

/* Solver mode.  NB_SOLVER_PARITY (default): the reference's exact Gauss-Seidel order (nudge.cpp:4206-4340 schedule, 4640-4855 sweeps),
 * bit-identical impulses.  NB_SOLVER_THROUGHPUT: mass-splitting Jacobi over the same constraint rows (nudge_b200/csrc/nb_jacobi.cuh) -
 * order independent, HBM-streaming, converges to the same contact problem but its impulses after N sweeps differ from the reference's
 * (validated by invariants and against a CPU restatement within a tolerance, tests/test_gpu_throughput.py).  Takes effect from the
 * next nb_setup_contact_constraints / nb_step.  The NB_SOLVER=throughput environment variable selects it at nb_create. */
enum nb_solver_mode { NB_SOLVER_PARITY = 0, NB_SOLVER_THROUGHPUT = 1 };
int nb_set_solver_mode(nb_context*, int mode);
int nb_get_solver_mode(const nb_context*);

/* CUDA-event timing of the dominant solver kernel across plain (non-graph) launches; see nb_api.cu. */
int nb_debug_timing_enable(nb_context*, int on);
int nb_debug_timing(nb_context*, uint32_t* launches, float* total_ms, void* stream);

/* Kernel-launch counter (every kernel this library launches increments it) and named device buffers for parity tests. */
uint64_t nb_launch_count(const nb_context*);
int nb_debug_read(nb_context*, const char* name, void* dst, size_t max_bytes, size_t* bytes, void* stream); /* synchronises */

int nb_debug_enable(nb_context*, int on);  /* keep the sorted broadphase pair list readable as "pair_keys" */
int nb_debug_sort(nb_context*, uint64_t* keys, uint32_t* vals /* may be null */, uint32_t n, int begin_bit, int end_bit); /* host pointers, in place */
int nb_debug_scan(nb_context*, uint32_t* data, uint32_t n, uint32_t* total);                                             /* exclusive scan, in place */

/* rcpps / rsqrtps model (SURVEY.md §0.5): tables are sampled from the host CPU in nb_create. */
int nb_debug_rcp(nb_context*, const float* x, float* y, uint32_t n, int rsqrt);  /* runs the device LUT path; host pointers */
int nb_lut_model_exact(const nb_context*);  /* 1 if the host CPU's rcpps/rsqrtps match the truncated-mantissa model on 2^20 probes */

#ifdef __cplusplus
}
#endif
#endif
