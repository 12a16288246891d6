// nudge_b200 — host side of the C ABI (include/nudge_b200.h): context, HBM arena, kernel sequencing.
// The reference keeps all memory caller-owned and bump-allocates scratch from an Arena (nudge.cpp:990-1055);
// here the context plays both roles for device memory: every buffer is carved once from cudaMalloc at
// nb_create and reused every step, nothing is allocated or synchronised inside the step.
#include "nb_shard.cuh"
#define NB_DEFAULT_COOP_LAUNCH 1
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>
#include <algorithm>
#include <math.h>
#include <nvtx3/nvToolsExt.h>

extern "C" void nb_host_sample_luts(u32* rcp_lut, u32* rsqrt_lut);   // nb_lut_host.cpp
extern "C" int nb_host_check_lut_model(const u32* rcp_lut, const u32* rsqrt_lut);


struct nb_context {
	nb_config cfg;
	int sms;
	std::string error;
	unsigned long long launches;
	int lut_exact;
	std::vector<void*> allocs;
	u32 B, nboxes, nspheres, nconn;  // uploaded sizes
	u32 tagbits, kbits, bodybits, batchbits;
	u32 stride;    // scratch stride
	u32 cstride;   // row plane stride
	u32 slots_per_bucket;
	int coop_blocks_solve; int coop_launch;
	u64* keybits;  // OR, AND of the Morton codes of the current collide
	bool defer_warm_start;  // nb_step: the warm start runs inside the first solver launch
	// nb_step as a CUDA graph: captured once per (stream, parameters, scene shape), replayed afterwards
	struct StepKey { cudaStream_t stream; float ts, gravity, damping; u32 iterations, B, nboxes, nspheres, nconn, tagbits, kbits; int debug, solver_mode; unsigned long long urow_version; } graph_key;
	cudaGraphExec_t graph_exec; unsigned long long graph_launches; int graph_enabled; bool capturing;
	int graph_is_coop;  // the recorded graph holds cooperative kernel nodes
	int graph_coop;  // 1: grid-synchronising kernels keep the cooperative-launch attribute inside the captured graph (co-residency guaranteed by the driver)
	u32* chain_start; u32* chain_len;  // per body: first entry / number of entries in the (body, batch) chain sort
	bool contacts_internal;  // the current contact set came from nb_collide (not nb_upload_contacts)
	u32 solve_backoff_ns;
	// throughput mode (nb_set_solver_mode): mass-splitting Jacobi, nb_jacobi.cuh
	int solver_mode; u32* jcnt; float4* jd; int jacobi_blocks1, jacobi_blocks2, jacobi_stages;
	// CUDA-event timing of the dominant solver kernel (nb_debug_timing): bench.py's roofline numerator is measured live
	int timing; cudaEvent_t tev[2][64]; int tev_n; bool tev_made;
	// nb_step overlaps independent branches of the step on a second stream (fork/join with events; also inside the captured graph)
	bool rows_on_side, join_before_solve, zero_chain_len; int overlap; cudaStream_t side; cudaEvent_t ev_fork, ev_fork2, ev_join, ev_join2; u32* flags2; u32* offs2; u32* block_sums2;
	// user constraint rows (nb_upload_constraint_rows, nb_rows_api.cuh)
	float4* instances;   // nb_instance_matrices with a host destination (allocated on first use)
	// nb_upload_bodies sends what the collision stage does not read (momentum, properties) on a second stream, so that copy runs under
	// `collide`; the first consumer waits for ev_up_done (inside a captured step: an external event-wait node, re-armed by every upload)
	cudaStream_t copy_stream; cudaEvent_t ev_up_begin, ev_up_done; bool upload_pending, capture_joined; int copy_overlap;
	int solve_wide;   // k_solve hands a body's row over with one 256-bit access instead of two 128-bit ones (default; NB_SOLVE_WIDE=0: the 128-bit protocol)
	nb_constraint_row* urows; u32 urow_cap, urow_n, urow_levels; unsigned long long urow_version; std::vector<u32> urow_level_off, urow_order;
	// ray-cast snapshot (nb_build_query_tree, nb_query_api.cuh): every buffer its own, allocated on first use, never one the step reads
	struct Query {
		bool built; u32 nboxes, nspheres, K;   // collider counts when the snapshot was taken (K = 0: empty scene)
		nb_transform* world_xf; float4* aabb_min; float4* aabb_max; u32* col_tag; u32* col_body; u32* counts; u64* keybits;
		u32* order; u32* rank; u64* mkeys; float4* tree_min; float4* tree_max; float4* leaf; SortBuffers sb; Tree T;
		nb_ray* rays; nb_ray_hit* hits; u32 io_cap;   // staging of host rays / hits
	} q;

	// scene
	nb_transform* xf; nb_body_properties* props; nb_body_momentum* mom; uint8_t* idle;
	u32* box_tags; nb_box_collider* box_data; nb_transform* box_xf;
	u32* sph_tags; nb_sphere_collider* sph_data; nb_transform* sph_xf;
	nb_body_pair* conn;
	u32* counts;
	// collide
	nb_transform* world_xf; float4* aabb_min; float4* aabb_max; u32* col_tag; u32* col_body; u32* order; u32* rank;
	float4* tree_min; float4* tree_max;
	u64* mkeys; uint8_t* smallf; u32* large_list; u64* table_keys; u64* table_vals; u32 table_mask; int use_tree;
	SortBuffers sb; u32 sort_cap;
	u64* pair_keys;  // alias into sb.keys[] after the pair sort
	u64* pair_keys_debug;  // copy kept for parity tests when debug is enabled (the sort buffers are reused later in the step)
	int debug;
	u32* flags; u32* offs; u32* block_sums;
	uint2* live; float* np_pen; u32* np_info; u32* np_list; u32* np_start;
	ContactOut staged, fin;
	u64* sleeping;
	u32* parent; u32* active; u32* active_idx; u32* taint;
	// cache
	u64* cache_tags; u32* cache_features; float4* cache_data;
	u64* culled_tags; u32* culled_features; float4* culled_data;
	u32* sorted; float4* impulses;
	// setup / solve
	float4* inertia;
	u32* sched_spill_ent; u32* sched_spill_uid; u32 sched_spill_cap;   // k_schedule's open-slot list beyond its on-chip positions
	u32* slot_of; u32* slot_done; u32* slot_left; u32* left_count; u32* batch_of; u32* slot_idx; float4* mw; uint2* cab; uint8_t* back;
	Rows rows;
};

#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { ctx->error = std::string(#call) + ": " + cudaGetErrorString(e_); return NB_ERR_CUDA; } } while (0)

template<class T>
static int dev_alloc(nb_context* ctx, T** p, size_t n) {
	void* q = nullptr;
	size_t bytes = (n ? n : 1) * sizeof(T);
	cudaError_t e = cudaMalloc(&q, bytes);
	if (e != cudaSuccess) { ctx->error = std::string("cudaMalloc: ") + cudaGetErrorString(e); return NB_ERR_CUDA; }
	cudaMemset(q, 0, bytes);
	ctx->allocs.push_back(q);
	*p = (T*)q;
	return 0;
}
#define ALLOC(p, n) do { int r_ = dev_alloc(ctx, &(p), (size_t)(n)); if (r_) return r_; } while (0)

static u32 bits_for(u64 n) { u32 b = 1; while (((u64)1 << b) < n) ++b; return b; }
static Launch mk_launch(nb_context* ctx, void* stream) { Launch L = { (cudaStream_t)stream, &ctx->launches, ctx->sms }; return L; }
#define GRID(n) nb_grid_for((unsigned)(n), ctx->sms)
// NVTX range per API call (SURVEY.md section 5): visible in Nsight timelines, a no-op costing tens of nanoseconds without a tool attached
struct NbRange { NbRange(const char* name) { nvtxRangePushA(name); } ~NbRange() { nvtxRangePop(); } };
#define NB_RANGE(name) NbRange nb_range_(name)
static int launch_user_rows(nb_context* ctx, int warm, cudaStream_t st);   // nb_rows_api.cuh

__global__ void k_reset_collide(u32* counts, u32 K, u64* keybits) {
	if (threadIdx.x == 0) {
		keybits[0] = 0; keybits[1] = ~(u64)0;
		counts[CNT_SCRATCH1] = K;  // key count of the Morton sort
		counts[CNT_PAIRS] = 0; counts[CNT_OVERFLOW] = 0; counts[CNT_EXT_SUM] = 0;
		for (int k = 0; k < 18; ++k) counts[CNT_EXT_HIST + k] = 0;
		for (int k = 0; k < 4; ++k) { counts[CNT_BMIN0 + k] = 0xffffffffu; counts[CNT_BMAX0 + k] = 0; }
	}
}
__global__ void __launch_bounds__(NB_BLOCK) k_copy_u64(const u64* src, u64* dst, const u32* n_ptr) {
	u32 n = *n_ptr;
	for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) dst[i] = src[i];
}
__global__ void __launch_bounds__(NB_BLOCK) k_copy_u32(const u32* src, u32* dst, const u32* n_ptr) {
	u32 n = *n_ptr;
	for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) dst[i] = src[i];
}
__global__ void __launch_bounds__(NB_BLOCK) k_debug_rcp(const float* x, float* y, u32 n, int rsq) {
	for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) y[i] = rsq ? nb_rsqrt(x[i]) : nb_rcp(x[i]);
}

// Ghost exchange for a scene sharded across GPUs (SURVEY.md §8e, K16): gather / scatter whole 32-byte BodyMomentum rows.
__global__ void __launch_bounds__(NB_BLOCK) k_pack_rows(const float4* rows, const u32* idx, u32 n, float4* out) {
	for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < 2 * n; i += gridDim.x * blockDim.x) out[i] = rows[2 * idx[i >> 1] + (i & 1)];
}
__global__ void __launch_bounds__(NB_BLOCK) k_unpack_rows(float4* rows, const u32* idx, const u32* src, u32 n, const float4* in) {
	for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < 2 * n; i += gridDim.x * blockDim.x) rows[2 * idx[i >> 1] + (i & 1)] = in[2 * src[i >> 1] + (i & 1)];
}

// Called by everything that touches momentum or properties on `st`: orders it after a pending nb_upload_bodies side copy.
static int join_uploads(nb_context* ctx, cudaStream_t st) {
	if (ctx->capturing) {   // in a captured step: one event-wait node that, at every replay, waits for the most recent upload's copy
		if (ctx->copy_stream && !ctx->capture_joined) { CK(cudaStreamWaitEvent(st, ctx->ev_up_done, cudaEventWaitExternal)); ctx->capture_joined = true; }
		return NB_OK;
	}
	if (ctx->upload_pending) { CK(cudaStreamWaitEvent(st, ctx->ev_up_done, 0)); ctx->upload_pending = false; }
	return NB_OK;
}
#define JOIN_UPLOADS() do { int r_ = join_uploads(ctx, (cudaStream_t)stream); if (r_) return r_; } while (0)

extern "C" {

int nb_pack_momentum(nb_context* ctx, const uint32_t* dev_indices, uint32_t n, void* dev_out, void* stream) {
	if (!n) return NB_OK;
	JOIN_UPLOADS();
	k_pack_rows<<<GRID(2 * n), NB_BLOCK, 0, (cudaStream_t)stream>>>((const float4*)ctx->mom, dev_indices, n, (float4*)dev_out);
	++ctx->launches;
	CK(cudaGetLastError());
	return NB_OK;
}
int nb_unpack_momentum(nb_context* ctx, const uint32_t* dev_indices, const uint32_t* dev_sources, uint32_t n, const void* dev_in, void* stream) {
	if (!n) return NB_OK;
	JOIN_UPLOADS();
	k_unpack_rows<<<GRID(2 * n), NB_BLOCK, 0, (cudaStream_t)stream>>>((float4*)ctx->mom, dev_indices, dev_sources, n, (const float4*)dev_in);
	++ctx->launches;
	CK(cudaGetLastError());
	return NB_OK;
}

int nb_create(const nb_config* config, nb_context** out) {
	if (!config || !out) return NB_ERR_ARGUMENT;
	nb_context* ctx = new nb_context();
	*out = ctx;
	ctx->cfg = *config;
	ctx->launches = 0;
	nb_config& c = ctx->cfg;
	if (!c.max_bodies) c.max_bodies = 1;
	u32 K = c.max_boxes + c.max_spheres;
	if (!c.max_pairs) c.max_pairs = 16 * (K ? K : 1);
	if (!c.max_contacts) c.max_contacts = 24 * c.max_bodies;
	int ndev = 0;
	CK(cudaGetDeviceCount(&ndev));
	if (ndev <= 0) { ctx->error = "no CUDA device: nudge_b200 has no CPU path"; return NB_ERR_CUDA; }
	CK(cudaSetDevice(c.device));
	cudaDeviceProp prop;
	CK(cudaGetDeviceProperties(&prop, c.device));
	ctx->sms = prop.multiProcessorCount;
	if (!prop.cooperativeLaunch) { ctx->error = "device lacks cooperative launch"; return NB_ERR_CUDA; }

	const u32 B = c.max_bodies, P = c.max_pairs, C = c.max_contacts;
	ctx->B = 0; ctx->nboxes = 0; ctx->nspheres = 0; ctx->nconn = 0;
	ctx->tagbits = 1; ctx->kbits = bits_for(K ? K : 1); ctx->bodybits = bits_for(B); ctx->batchbits = bits_for((u64)C + 2);
	ctx->stride = ((std::max(std::max(P, C), std::max(B, K)) + 63) / 64) * 64;
	ctx->cstride = ((C + 8 * 16 * NB_SCHED_MAXV + 31) / 32) * 32;  // slots = batch*8 + lane; leftover batches of the 16 buckets may be partly empty (a hub body beyond that: OVF_SCHED from k_batch_index)
	ctx->slots_per_bucket = (C + 15) / 16 + 1;

	ALLOC(ctx->xf, B); ALLOC(ctx->props, B); ALLOC(ctx->mom, B); ALLOC(ctx->idle, B);
	ALLOC(ctx->box_tags, c.max_boxes); ALLOC(ctx->box_data, c.max_boxes); ALLOC(ctx->box_xf, c.max_boxes);
	ALLOC(ctx->sph_tags, c.max_spheres); ALLOC(ctx->sph_data, c.max_spheres); ALLOC(ctx->sph_xf, c.max_spheres);
	ALLOC(ctx->conn, c.max_connections);
	ALLOC(ctx->counts, CNT__COUNT); ALLOC(ctx->keybits, 2);
	ALLOC(ctx->world_xf, K); ALLOC(ctx->aabb_min, K); ALLOC(ctx->aabb_max, K); ALLOC(ctx->col_tag, K); ALLOC(ctx->col_body, K);
	ALLOC(ctx->order, K); ALLOC(ctx->rank, K);
	size_t tree_nodes = 0; { u32 n = K ? K : 1; tree_nodes = n; while (n > 8) { n = (n + 7) / 8; tree_nodes += n; } }
	ALLOC(ctx->tree_min, tree_nodes + 8); ALLOC(ctx->tree_max, tree_nodes + 8);
	{
		u32 tsz = 1024; while (tsz < 2 * (K ? K : 1)) tsz *= 2;
		ctx->table_mask = tsz - 1;
		ALLOC(ctx->mkeys, K); ALLOC(ctx->smallf, K); ALLOC(ctx->large_list, K); ALLOC(ctx->table_keys, tsz); ALLOC(ctx->table_vals, tsz);
		const char* e = getenv("NB_BROADPHASE");
		ctx->use_tree = e && !strcmp(e, "tree");
	}
	ctx->sort_cap = std::max(std::max(K, P), 2 * C);
	for (int i = 0; i < 2; ++i) { ALLOC(ctx->sb.keys[i], ctx->sort_cap); ALLOC(ctx->sb.vals[i], ctx->sort_cap); }
	ALLOC(ctx->sb.hist, 256 * NB_SORT_GRID);
	ctx->sb.bar = ctx->counts + CNT_BAR0;
	{ const char* e = getenv("NB_SORT"); ctx->sb.coop_blocks = (e && !strcmp(e, "legacy")) ? 0 : ctx->sms; }
	// Grid-synchronising kernels (one block per SM for the sort, the occupancy-derived grid for the solver) are launched as
	// ordinary kernels unless NB_COOP_LAUNCH=1: the grid fits the idle device by construction, and a cooperative launch costs
	// several microseconds more per launch.
	{ const char* e = getenv("NB_GRAPH"); ctx->graph_enabled = e ? atoi(e) != 0 : 1; }
	{ const char* e = getenv("NB_GRAPH_COOP"); ctx->graph_coop = e ? atoi(e) != 0 : 1; }
	{ const char* e = getenv("NB_COOP_LAUNCH"); ctx->coop_launch = e ? atoi(e) != 0 : NB_DEFAULT_COOP_LAUNCH; ctx->sb.coop_launch = ctx->coop_launch; }
	CK(cudaFuncSetAttribute(k_sort_coop<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(CoopSortSmem)));
	CK(cudaFuncSetAttribute(k_sort_coop<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(CoopSortSmem))); ALLOC(ctx->sb.block_sums, 8 * NB_SCAN_GRID);
	ALLOC(ctx->flags, 5 * (size_t)ctx->stride); ALLOC(ctx->offs, 5 * (size_t)ctx->stride); ALLOC(ctx->block_sums, 16 * NB_SCAN_GRID);
	{ const char* e = getenv("NB_SCAN"); g_nb_scan_three_kernels = !(e && !strcmp(e, "single")); }  // the single-launch variant measured slower (profiles/)
	ALLOC(ctx->live, P); ALLOC(ctx->np_pen, P); ALLOC(ctx->np_info, P); ALLOC(ctx->np_list, P); ALLOC(ctx->np_start, P);
	ALLOC(ctx->staged.data, 2 * (size_t)C); ALLOC(ctx->staged.bodies, C); ALLOC(ctx->staged.tags, C); ALLOC(ctx->staged.features, C);
	ALLOC(ctx->fin.data, 2 * (size_t)C); ALLOC(ctx->fin.bodies, C); ALLOC(ctx->fin.tags, C); ALLOC(ctx->fin.features, C);
	ALLOC(ctx->sleeping, (size_t)P + C);
	ALLOC(ctx->parent, B); ALLOC(ctx->active, B); ALLOC(ctx->active_idx, B); ALLOC(ctx->taint, B);
	ALLOC(ctx->cache_tags, C); ALLOC(ctx->cache_features, C); ALLOC(ctx->cache_data, C);
	ALLOC(ctx->culled_tags, C); ALLOC(ctx->culled_features, C); ALLOC(ctx->culled_data, C);
	ALLOC(ctx->sorted, C); ALLOC(ctx->impulses, C);
	ALLOC(ctx->inertia, 2 * (size_t)B);
	ALLOC(ctx->slot_of, C); ALLOC(ctx->slot_done, 16 * (size_t)ctx->slots_per_bucket); ALLOC(ctx->slot_left, 16 * (size_t)ctx->slots_per_bucket);
	ctx->sched_spill_cap = std::min<u32>(ctx->slots_per_bucket + 2, 16384u);
	ALLOC(ctx->sched_spill_ent, 16 * (size_t)ctx->sched_spill_cap * 16); ALLOC(ctx->sched_spill_uid, 16 * (size_t)ctx->sched_spill_cap);
	CK(cudaMemset(ctx->sched_spill_ent, 0xff, sizeof(u32) * 16 * (size_t)ctx->sched_spill_cap * 16));
	ALLOC(ctx->left_count, 16); ALLOC(ctx->batch_of, C); ALLOC(ctx->slot_idx, C); ALLOC(ctx->mw, 2 * (size_t)B); ALLOC(ctx->cab, C); ALLOC(ctx->back, C);
	ALLOC(ctx->rows.plane, (size_t)ROW_PLANES_TOTAL * ctx->cstride); ALLOC(ctx->rows.state, 3 * (size_t)ctx->cstride);
	ALLOC(ctx->rows.a, ctx->cstride); ALLOC(ctx->rows.b, ctx->cstride); ALLOC(ctx->rows.contact, ctx->cstride); ALLOC(ctx->rows.wait, 2 * (size_t)ctx->cstride); ALLOC(ctx->chain_start, B); ALLOC(ctx->chain_len, B);
	ctx->rows.stride = ctx->cstride;
	ALLOC(ctx->jcnt, B); ALLOC(ctx->jd, 2 * (size_t)B);
	ALLOC(ctx->flags2, ctx->stride); ALLOC(ctx->offs2, ctx->stride); ALLOC(ctx->block_sums2, 16 * NB_SCAN_GRID);
	// measured (profiles/r02b): 1.277 ms per step with the two branches on the second stream, 1.275 ms without — the branches are
	// short next to the sort / scheduler they run beside and the extra graph edges cost what they save.  Kept opt-in (NB_OVERLAP=1).
	{ const char* e = getenv("NB_OVERLAP"); ctx->overlap = e ? atoi(e) != 0 : 0; }
	CK(cudaStreamCreateWithFlags(&ctx->side, cudaStreamNonBlocking));
	CK(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&ctx->ev_fork2, cudaEventDisableTiming));
	CK(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&ctx->ev_join2, cudaEventDisableTiming));
	// upload of the rows `collide` does not read, on a copy stream of its own (NB_COPY_OVERLAP=0: everything on the caller's stream)
	{ const char* e = getenv("NB_SOLVE_WIDE"); ctx->solve_wide = e ? atoi(e) != 0 : 1; }   // measured: 0.492 -> 0.419 ms per launch on the 64k pile (profiles/r02r_*)
	{ const char* e = getenv("NB_COPY_OVERLAP"); ctx->copy_overlap = e ? atoi(e) != 0 : 1; }
	CK(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
	CK(cudaEventCreateWithFlags(&ctx->ev_up_begin, cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&ctx->ev_up_done, cudaEventDisableTiming));
	CK(cudaEventRecord(ctx->ev_up_done, ctx->copy_stream));   // a first, already complete record for the step graph's event-wait node
	ctx->solver_mode = NB_SOLVER_PARITY;
	CK(cudaFuncSetAttribute(k_jacobi_sweep<true, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(JacobiSmem<1>)));
	CK(cudaFuncSetAttribute(k_jacobi_sweep<false, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(JacobiSmem<1>)));
	CK(cudaFuncSetAttribute(k_jacobi_sweep<true, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(JacobiSmem<2>)));
	CK(cudaFuncSetAttribute(k_jacobi_sweep<false, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(JacobiSmem<2>)));
	{
		int per1 = 0, per2 = 0;
		CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per1, k_jacobi_sweep<false, 1>, NJ_TILE, sizeof(JacobiSmem<1>)));
		CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per2, k_jacobi_sweep<false, 2>, NJ_TILE, sizeof(JacobiSmem<2>)));
		if (per1 < 1 || per2 < 1) { ctx->error = "k_jacobi_sweep does not fit on an SM"; return NB_ERR_CUDA; }
		ctx->jacobi_blocks1 = ctx->sms * per1; ctx->jacobi_blocks2 = ctx->sms * per2;   // persistent: every CTA walks tiles blockIdx.x, + gridDim.x, ...
		ctx->jacobi_stages = 0;   // 0 = by body count at launch
		if (const char* e = getenv("NB_JACOBI_STAGES")) ctx->jacobi_stages = atoi(e);
		if (const char* e = getenv("NB_SOLVER")) ctx->solver_mode = !strcmp(e, "throughput") ? NB_SOLVER_THROUGHPUT : NB_SOLVER_PARITY;
	}
	ctx->pair_keys = ctx->sb.keys[0];
	ctx->pair_keys_debug = nullptr; ctx->debug = 0;

	// rcpps / rsqrtps tables from this host's CPU (SURVEY.md §0.5)
	u32 rcp_lut[2048], rsqrt_lut[2048];
	nb_host_sample_luts(rcp_lut, rsqrt_lut);
	ctx->lut_exact = nb_host_check_lut_model(rcp_lut, rsqrt_lut);
	CK(cudaMemcpyToSymbol(c_rcp_lut, rcp_lut, sizeof(rcp_lut)));
	CK(cudaMemcpyToSymbol(c_rsqrt_lut, rsqrt_lut, sizeof(rsqrt_lut)));
	CK(cudaMemcpyToSymbol(g_rcp_lut, rcp_lut, sizeof(rcp_lut)));
	CK(cudaMemcpyToSymbol(g_rsqrt_lut, rsqrt_lut, sizeof(rsqrt_lut)));

	int per_sm = 0;
	CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_solve<false>, NB_BLOCK, 0));
	if (per_sm < 1) { ctx->error = "k_solve does not fit on an SM"; return NB_ERR_CUDA; }
	if (const char* e = getenv("NB_SOLVE_BLOCKS_PER_SM")) { int v = atoi(e); if (v >= 1 && v < per_sm) per_sm = v; }
	ctx->solve_backoff_ns = 150;  // sleep per missing application while a contact is >= 2 applications away (nanosleep may take up to 2x)
	if (const char* e = getenv("NB_SOLVE_HOP_NS")) ctx->solve_backoff_ns = (u32)atoi(e);
	ctx->coop_blocks_solve = ctx->sms * per_sm;  // all co-resident: the dataflow solver relies on it
	CK(cudaDeviceSynchronize());
	return NB_OK;
}

void nb_destroy(nb_context* ctx) {
	if (!ctx) return;
	cudaDeviceSynchronize();
	if (ctx->graph_exec) cudaGraphExecDestroy(ctx->graph_exec);
	if (ctx->tev_made) for (int i = 0; i < 64; ++i) { cudaEventDestroy(ctx->tev[0][i]); cudaEventDestroy(ctx->tev[1][i]); }
	if (ctx->copy_stream) { cudaStreamDestroy(ctx->copy_stream); cudaEventDestroy(ctx->ev_up_begin); cudaEventDestroy(ctx->ev_up_done); }
	if (ctx->side) { cudaStreamDestroy(ctx->side); cudaEventDestroy(ctx->ev_fork); cudaEventDestroy(ctx->ev_fork2); cudaEventDestroy(ctx->ev_join); cudaEventDestroy(ctx->ev_join2); }
	for (size_t i = 0; i < ctx->allocs.size(); ++i) cudaFree(ctx->allocs[i]);
	delete ctx;
}

const char* nb_last_error(const nb_context* ctx) { return ctx ? ctx->error.c_str() : "null context"; }
uint64_t nb_launch_count(const nb_context* ctx) { return ctx->launches; }
int nb_lut_model_exact(const nb_context* ctx) { return ctx->lut_exact; }

#define H2D(dst, src, n, T) CK(cudaMemcpyAsync(dst, src, (size_t)(n) * sizeof(T), cudaMemcpyHostToDevice, (cudaStream_t)stream))
#define D2H(dst, src, n, T) CK(cudaMemcpyAsync(dst, src, (size_t)(n) * sizeof(T), cudaMemcpyDeviceToHost, (cudaStream_t)stream))

int nb_upload_bodies(nb_context* ctx, const nb_body_data* h, void* stream) {
	NB_RANGE("nb_upload_bodies");
	if (h->count > ctx->cfg.max_bodies) { ctx->error = "too many bodies"; return NB_ERR_CAPACITY; }
	ctx->B = h->count;
	cudaStream_t st = (cudaStream_t)stream;
	H2D(ctx->xf, h->transforms, h->count, nb_transform); H2D(ctx->idle, h->idle_counters, h->count, uint8_t);   // all the collision stage reads
	if (ctx->copy_overlap && ctx->copy_stream && st != nullptr && st != cudaStreamLegacy && st != cudaStreamPerThread) {
		CK(cudaEventRecord(ctx->ev_up_begin, st));                       // after everything already queued on the caller's stream (it may still use the old rows)
		CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_up_begin, 0));
		CK(cudaMemcpyAsync(ctx->mom, h->momentum, (size_t)h->count * sizeof(nb_body_momentum), cudaMemcpyHostToDevice, ctx->copy_stream));
		CK(cudaMemcpyAsync(ctx->props, h->properties, (size_t)h->count * sizeof(nb_body_properties), cudaMemcpyHostToDevice, ctx->copy_stream));
		CK(cudaEventRecord(ctx->ev_up_done, ctx->copy_stream));
		ctx->upload_pending = true;
	}
	else {
		H2D(ctx->props, h->properties, h->count, nb_body_properties); H2D(ctx->mom, h->momentum, h->count, nb_body_momentum);
	}
	return NB_OK;
}
#define ROWS_OK(count) do { if ((count) > ctx->cfg.max_bodies) { ctx->error = "row count exceeds max_bodies"; return NB_ERR_CAPACITY; } } while (0)
int nb_upload_momentum(nb_context* ctx, const nb_body_momentum* h, uint32_t count, void* stream) { ROWS_OK(count); JOIN_UPLOADS(); H2D(ctx->mom, h, count, nb_body_momentum); return NB_OK; }
int nb_upload_transforms(nb_context* ctx, const nb_transform* h, uint32_t count, void* stream) { ROWS_OK(count); H2D(ctx->xf, h, count, nb_transform); return NB_OK; }
int nb_download_momentum(nb_context* ctx, nb_body_momentum* h, uint32_t count, void* stream) { ROWS_OK(count); JOIN_UPLOADS(); D2H(h, ctx->mom, count, nb_body_momentum); return NB_OK; }
int nb_download_transforms(nb_context* ctx, nb_transform* h, uint32_t count, void* stream) { ROWS_OK(count); D2H(h, ctx->xf, count, nb_transform); return NB_OK; }

int nb_upload_colliders(nb_context* ctx, const nb_collider_data* h, void* stream) {
	if (h->boxes.count > ctx->cfg.max_boxes || h->spheres.count > ctx->cfg.max_spheres) { ctx->error = "too many colliders"; return NB_ERR_CAPACITY; }
	ctx->nboxes = h->boxes.count; ctx->nspheres = h->spheres.count;
	u32 maxtag = 1;
	for (u32 i = 0; i < h->boxes.count; ++i) maxtag = std::max(maxtag, h->boxes.tags[i]);
	for (u32 i = 0; i < h->spheres.count; ++i) maxtag = std::max(maxtag, h->spheres.tags[i]);
	ctx->tagbits = bits_for((u64)maxtag + 1);
	ctx->kbits = bits_for(std::max(1u, ctx->nboxes + ctx->nspheres));
	H2D(ctx->box_tags, h->boxes.tags, h->boxes.count, u32); H2D(ctx->box_data, h->boxes.data, h->boxes.count, nb_box_collider);
	H2D(ctx->box_xf, h->boxes.transforms, h->boxes.count, nb_transform);
	H2D(ctx->sph_tags, h->spheres.tags, h->spheres.count, u32); H2D(ctx->sph_data, h->spheres.data, h->spheres.count, nb_sphere_collider);
	H2D(ctx->sph_xf, h->spheres.transforms, h->spheres.count, nb_transform);
	return NB_OK;
}
int nb_upload_connections(nb_context* ctx, const nb_body_connections* h, void* stream) {
	if (h->count > ctx->cfg.max_connections) { ctx->error = "too many connections"; return NB_ERR_CAPACITY; }
	ctx->nconn = h->count;
	H2D(ctx->conn, h->data, h->count, nb_body_pair);
	return NB_OK;
}
int nb_upload_cache(nb_context* ctx, const nb_contact_cache* h, void* stream) {
	if (h->count > ctx->cfg.max_contacts) { ctx->error = "cache too large"; return NB_ERR_CAPACITY; }
	H2D(ctx->cache_tags, h->tags, h->count, u64); H2D(ctx->cache_features, h->features, h->count, u32); H2D(ctx->cache_data, h->data, h->count, nb_cached_impulse);
	u32 n = h->count;
	CK(cudaMemcpyAsync(ctx->counts + CNT_CACHE, &n, 4, cudaMemcpyHostToDevice, (cudaStream_t)stream));
	CK(cudaStreamSynchronize((cudaStream_t)stream));
	return NB_OK;
}
int nb_download_bodies(nb_context* ctx, nb_body_data* h, void* stream) {
	NB_RANGE("nb_download_bodies");
	u32 n = std::min(h->count, ctx->B);
	JOIN_UPLOADS();
	D2H(h->transforms, ctx->xf, n, nb_transform); D2H(h->momentum, ctx->mom, n, nb_body_momentum); D2H(h->idle_counters, ctx->idle, n, uint8_t);
	CK(cudaStreamSynchronize((cudaStream_t)stream));
	return NB_OK;
}
static int get_counts(nb_context* ctx, u32* host, void* stream) {
	D2H(host, ctx->counts, CNT__COUNT, u32);
	CK(cudaStreamSynchronize((cudaStream_t)stream));
	return NB_OK;
}
int nb_download_counts(nb_context* ctx, nb_counts* out, void* stream) {
	u32 h[CNT__COUNT];
	int r = get_counts(ctx, h, stream); if (r) return r;
	out->pairs = h[CNT_PAIRS]; out->live_pairs = h[CNT_LIVE_TOTAL]; out->contacts = h[CNT_CONTACTS]; out->sleeping = h[CNT_SLEEPING];
	out->active = h[CNT_ACTIVE]; out->cache = h[CNT_CACHE]; out->culled = h[CNT_CULLED]; out->batches = h[CNT_BATCHES]; out->levels = h[CNT_LEVELS];
	out->overflow = h[CNT_OVERFLOW];
	if (h[CNT_OVERFLOW]) { ctx->error = "capacity overflow during the last step (nb_counts.overflow: 1 pairs, 2 contacts, 4 batch scheduler)"; return NB_ERR_OVERFLOW; }
	return NB_OK;
}
int nb_download_contacts(nb_context* ctx, nb_contact_data* h, nb_active_bodies* ha, void* stream) {
	u32 c[CNT__COUNT];
	int r = get_counts(ctx, c, stream); if (r) return r;
	if (h) {
		u32 n = c[CNT_CONTACTS], s = c[CNT_SLEEPING];
		if (n > h->capacity) { ctx->error = "host contact buffer too small"; return NB_ERR_CAPACITY; }
		// sleeping pairs can number up to the broadphase pairs; the reference sizes that buffer like the contact arrays (nudge.h:73-82)
		if (h->sleeping_pairs && s > h->capacity) { ctx->error = "host sleeping-pair buffer too small (it is bounded by nb_contact_data.capacity)"; return NB_ERR_CAPACITY; }
		h->count = n; h->sleeping_count = s;
		D2H(h->data, ctx->fin.data, n, nb_contact); D2H(h->bodies, ctx->fin.bodies, n, nb_body_pair);
		D2H(h->tags, ctx->fin.tags, n, u64); D2H(h->features, ctx->fin.features, n, u32);
		if (h->sleeping_pairs) D2H(h->sleeping_pairs, ctx->sleeping, s, u64);
	}
	if (ha) {
		u32 n = c[CNT_ACTIVE];
		if (n > ha->capacity) { ctx->error = "host active-body buffer too small"; return NB_ERR_CAPACITY; }
		ha->count = n;
		D2H(ha->indices, ctx->active_idx, n, u32);
	}
	CK(cudaStreamSynchronize((cudaStream_t)stream));
	return c[CNT_OVERFLOW] ? NB_ERR_OVERFLOW : NB_OK;
}
// Host -> HBM for the outputs of collide (the reference lets user code add or edit contacts between the calls, example/main.cpp:288).
int nb_upload_contacts(nb_context* ctx, const nb_contact_data* h, const nb_active_bodies* ha, void* stream) {
	if (h) {
		if (h->count > ctx->cfg.max_contacts || h->sleeping_count > ctx->cfg.max_contacts) { ctx->error = "too many contacts"; return NB_ERR_CAPACITY; }
		ctx->contacts_internal = false;
		H2D(ctx->fin.data, h->data, h->count, nb_contact); H2D(ctx->fin.bodies, h->bodies, h->count, nb_body_pair);
		H2D(ctx->fin.tags, h->tags, h->count, u64); H2D(ctx->fin.features, h->features, h->count, u32);
		if (h->sleeping_count) H2D(ctx->sleeping, h->sleeping_pairs, h->sleeping_count, u64);
		u32 n[2] = { h->count, h->sleeping_count };
		CK(cudaMemcpyAsync(ctx->counts + CNT_CONTACTS, &n[0], 4, cudaMemcpyHostToDevice, (cudaStream_t)stream));
		CK(cudaMemcpyAsync(ctx->counts + CNT_SLEEPING, &n[1], 4, cudaMemcpyHostToDevice, (cudaStream_t)stream));
	}
	if (ha) {
		if (ha->count > ctx->cfg.max_bodies) { ctx->error = "too many active bodies"; return NB_ERR_CAPACITY; }
		H2D(ctx->active_idx, ha->indices, ha->count, u32);
		u32 n = ha->count;
		CK(cudaMemcpyAsync(ctx->counts + CNT_ACTIVE, &n, 4, cudaMemcpyHostToDevice, (cudaStream_t)stream));
	}
	CK(cudaStreamSynchronize((cudaStream_t)stream));
	return NB_OK;
}

int nb_download_cache(nb_context* ctx, nb_contact_cache* h, void* stream) {
	u32 c[CNT__COUNT];
	int r = get_counts(ctx, c, stream); if (r) return r;
	u32 n = c[CNT_CACHE];
	if (n > h->capacity) { ctx->error = "host cache buffer too small"; return NB_ERR_CAPACITY; }
	h->count = n;
	D2H(h->tags, ctx->cache_tags, n, u64); D2H(h->features, ctx->cache_features, n, u32); D2H(h->data, ctx->cache_data, n, nb_cached_impulse);
	CK(cudaStreamSynchronize((cudaStream_t)stream));
	return NB_OK;
}

// ---------------- collide ----------------
int nb_collide(nb_context* ctx, void* stream) {
	NB_RANGE("nb_collide");
	Launch L = mk_launch(ctx, stream);
	cudaStream_t st = L.stream;
	const u32 K = ctx->nboxes + ctx->nspheres, B = ctx->B, nboxes = ctx->nboxes;
	u32* counts = ctx->counts;
	k_reset_collide<<<1, 32, 0, st>>>(counts, K, ctx->keybits); ++ctx->launches;
	if (K == 0 || B == 0) return NB_OK;
	k_collider_world<<<GRID(K), NB_BLOCK, 0, st>>>(ctx->nboxes, ctx->nspheres, ctx->xf, ctx->box_xf, ctx->box_data, ctx->box_tags,
		ctx->sph_xf, ctx->sph_data, ctx->sph_tags, ctx->world_xf, ctx->aabb_min, ctx->aabb_max, ctx->col_tag, ctx->col_body, counts);
	k_morton<<<GRID(K), NB_BLOCK, 0, st>>>(K, ctx->aabb_min, ctx->aabb_max, counts, ctx->sb.keys[0], ctx->sb.vals[0], ctx->keybits);
	ctx->launches += 2;
	// radix sort on the 48-bit code; ties keep index order like the stable sort of nudge.cpp:3165
	int cur = nb_radix_sort(L, ctx->sb, counts + CNT_SCRATCH1, 0, 48, true, 0, 0, 0, ctx->keybits);
	Tree T;
	{
		size_t off = 0; u32 n = K; int l = 0;
		while (true) { T.mn[l] = ctx->tree_min + off; T.mx[l] = ctx->tree_max + off; T.n[l] = n; off += n; ++l; if (n <= 8) break; n = (n + 7) / 8; }
		T.levels = l;
	}
	k_leaves<<<GRID(K), NB_BLOCK, 0, st>>>(K, ctx->sb.vals[cur], ctx->sb.keys[cur], ctx->aabb_min, ctx->aabb_max, ctx->order, ctx->rank, (float4*)T.mn[0], (float4*)T.mx[0], ctx->mkeys);
	++ctx->launches;
	if (ctx->use_tree) {  // NB_BROADPHASE=tree: the implicit 8-ary AABB tree (kept for comparison)
		for (int l = 1; l < T.levels; ++l) {
			k_build_level<<<GRID(T.n[l]), NB_BLOCK, 0, st>>>(T.mn[l - 1], T.mx[l - 1], T.n[l - 1], (float4*)T.mn[l], (float4*)T.mx[l], T.n[l]);
			++ctx->launches;
		}
		k_find_pairs<<<GRID(K), NB_BLOCK, 0, st>>>(T, K, ctx->order, ctx->kbits, ctx->sb.keys[0], ctx->cfg.max_pairs, counts);
		++ctx->launches;
	}
	else {
		CK(cudaMemsetAsync(ctx->table_keys, 0xff, sizeof(u64) * ((size_t)ctx->table_mask + 1), st));
		k_grid_setup<<<1, 1, 0, st>>>(K, counts);
		k_grid_build<<<GRID(K), NB_BLOCK, 0, st>>>(K, ctx->order, (float4*)T.mn[0], T.mx[0], ctx->mkeys, ctx->smallf, ctx->large_list, ctx->table_keys, ctx->table_vals, ctx->table_mask, counts);
		k_grid_pairs<<<GRID((size_t)K * 32), NB_BLOCK, 0, st>>>(K, ctx->order, T.mn[0], T.mx[0], ctx->smallf, ctx->mkeys, ctx->table_keys, ctx->table_vals, ctx->table_mask, ctx->kbits, ctx->sb.keys[0], ctx->cfg.max_pairs, counts);
		k_large_pairs<<<GRID(K), NB_BLOCK, 0, st>>>(K, ctx->order, T.mn[0], T.mx[0], ctx->smallf, ctx->large_list, ctx->kbits, ctx->sb.keys[0], ctx->cfg.max_pairs, counts);
		ctx->launches += 4;
	}
	k_clamp_count<<<1, 1, 0, st>>>(counts, CNT_PAIRS, ctx->cfg.max_pairs);
	++ctx->launches;
	cur = nb_radix_sort(L, ctx->sb, counts + CNT_PAIRS, 0, (int)(2 * ctx->kbits), false, 0);  // nudge.cpp:3498
	ctx->pair_keys = ctx->sb.keys[cur];
	if (ctx->debug) { k_copy_u64<<<GRID(ctx->cfg.max_pairs), NB_BLOCK, 0, st>>>(ctx->pair_keys, ctx->pair_keys_debug, counts + CNT_PAIRS); ++ctx->launches; }

	// coarse islands (nudge.cpp:3500-3703)
	const u32 P = ctx->cfg.max_pairs, S = ctx->stride;
	k_uf_init<<<GRID(B), NB_BLOCK, 0, st>>>(ctx->parent, ctx->active, ctx->taint, B); ++ctx->launches;
	if (ctx->nconn) { k_uf_union_conn<<<GRID(ctx->nconn), NB_BLOCK, 0, st>>>(ctx->parent, ctx->taint, ctx->idle, ctx->conn, ctx->nconn); ++ctx->launches; }
	k_uf_union_pairs<<<GRID(P), NB_BLOCK, 0, st>>>(ctx->parent, ctx->taint, ctx->idle, ctx->pair_keys, ctx->kbits, ctx->col_body, counts);
	k_uf_flatten_active<<<GRID(B), NB_BLOCK, 0, st>>>(ctx->parent, ctx->active, ctx->taint, ctx->idle, B);
	k_pair_flags<<<GRID(P), NB_BLOCK, 0, st>>>(ctx->pair_keys, ctx->kbits, nboxes, ctx->col_body, ctx->parent, ctx->active, ctx->flags, S, counts);
	ctx->launches += 3;
	nb_scan<5>(L, ctx->flags, ctx->offs, S, counts + CNT_PAIRS, 0, ctx->block_sums, counts + CNT_LIVE0);  // -> LIVE0..3, SLEEP_COARSE
	k_partition<<<GRID(P), NB_BLOCK, 0, st>>>(ctx->pair_keys, ctx->kbits, ctx->flags, ctx->offs, S, ctx->col_tag, ctx->live, ctx->sleeping, counts);
	++ctx->launches;

	// narrowphase: count, scan, emit (nudge.cpp:3753-3786)
	k_np_faces<<<GRID(P), NB_BLOCK, 0, st>>>(ctx->live, nboxes, ctx->world_xf, ctx->box_data, ctx->sph_data, ctx->col_tag, ctx->flags, S, ctx->np_pen, ctx->np_info, counts);
	++ctx->launches;
	nb_scan<1>(L, ctx->flags + 3 * (size_t)S, ctx->offs + 3 * (size_t)S, S, counts + CNT_LIVE0, 0, ctx->block_sums, counts + CNT_SURV);
	k_np_list<<<GRID(P), NB_BLOCK, 0, st>>>(ctx->flags, ctx->offs, S, ctx->np_list, counts);
	k_np_clip<<<GRID(P), NB_BLOCK, 0, st>>>(ctx->live, ctx->np_list, ctx->np_pen, ctx->np_info, ctx->world_xf, ctx->box_data, ctx->col_tag, ctx->flags, S,
		ctx->fin /* scratch: rewritten by k_contact_compact below */, ctx->np_start, ctx->cfg.max_contacts, counts);
	ctx->launches += 2;
	nb_scan<3>(L, ctx->flags, ctx->offs, S, counts + CNT_LIVE_TOTAL, 0, ctx->block_sums, counts + CNT_FACE);  // -> FACE, EDGE, OTHER
	k_np_emit<<<GRID(P), NB_BLOCK, 0, st>>>(ctx->live, ctx->np_list, ctx->np_start, ctx->fin, nboxes, ctx->world_xf, ctx->box_data, ctx->sph_data, ctx->col_tag,
		ctx->flags, ctx->offs, S, ctx->staged, ctx->cfg.max_contacts, counts);
	++ctx->launches;

	// fine islands, active bodies, contact compaction (nudge.cpp:3788-4006)
	const u32 C = ctx->cfg.max_contacts;
	k_uf_init<<<GRID(B), NB_BLOCK, 0, st>>>(ctx->parent, ctx->active, ctx->taint, B); ++ctx->launches;
	if (ctx->nconn) { k_uf_union_conn<<<GRID(ctx->nconn), NB_BLOCK, 0, st>>>(ctx->parent, ctx->taint, ctx->idle, ctx->conn, ctx->nconn); ++ctx->launches; }
	k_uf_union_contacts<<<GRID(C), NB_BLOCK, 0, st>>>(ctx->parent, ctx->taint, ctx->idle, ctx->staged.bodies, counts);
	k_uf_flatten_active<<<GRID(B), NB_BLOCK, 0, st>>>(ctx->parent, ctx->active, ctx->taint, ctx->idle, B);
	k_body_flags<<<GRID(B), NB_BLOCK, 0, st>>>(ctx->parent, ctx->active, ctx->flags, B);
	ctx->launches += 3;
	nb_scan<1>(L, ctx->flags, ctx->offs, S, nullptr, B, ctx->block_sums, counts + CNT_ACTIVE);
	k_active_scatter<<<GRID(B), NB_BLOCK, 0, st>>>(ctx->flags, ctx->offs, ctx->active_idx, B);
	k_contact_flags<<<GRID(C), NB_BLOCK, 0, st>>>(ctx->staged.bodies, ctx->staged.tags, ctx->parent, ctx->active, ctx->flags, S, counts);
	ctx->launches += 2;
	nb_scan<2>(L, ctx->flags, ctx->offs, S, counts + CNT_STAGED, 0, ctx->block_sums, counts + CNT_CONTACTS);  // -> CONTACTS, SLEEP_FINE
	k_contact_compact<<<GRID(C), NB_BLOCK, 0, st>>>(ctx->staged, ctx->fin, ctx->flags, ctx->offs, S, ctx->sleeping, counts);
	++ctx->launches;

	// sort sleeping pairs (nudge.cpp:4008): key X | Y<<32, both below 2^tagbits
	k_copy_u64<<<GRID(C), NB_BLOCK, 0, st>>>(ctx->sleeping, ctx->sb.keys[0], counts + CNT_SLEEPING); ++ctx->launches;
	cur = nb_radix_sort(L, ctx->sb, counts + CNT_SLEEPING, 0, (int)ctx->tagbits, false, 0, 32, (int)(32 + ctx->tagbits));
	k_copy_u64<<<GRID(C), NB_BLOCK, 0, st>>>(ctx->sb.keys[cur], ctx->sleeping, counts + CNT_SLEEPING); ++ctx->launches;
	ctx->contacts_internal = true;
	CK(cudaGetLastError());
	return NB_OK;
}

int nb_apply_gravity_damping(nb_context* ctx, float time_step, float gravity, float damping, void* stream) {
	NB_RANGE("nb_apply_gravity_damping");
	JOIN_UPLOADS();   // first reader of the momentum rows in a step
	k_gravity_damping<<<GRID(ctx->B), NB_BLOCK, 0, (cudaStream_t)stream>>>(ctx->active_idx, ctx->mom, time_step, gravity, damping, ctx->counts);
	++ctx->launches;
	CK(cudaGetLastError());
	return NB_OK;
}

// ---------------- contact cache ----------------
// The two halves of read_cached_impulses are independent of each other: (a) the tag ORDER of the contacts (one sort), (b) the cache
// LOOKUP of every contact's impulse plus the entries of sleeping pairs that survive the frame.  nb_step runs (b) on a second stream.
static int read_lookup(nb_context* ctx, cudaStream_t st, u32* flags, u32* offs, u32* block_sums) {
	Launch L = { st, &ctx->launches, ctx->sms };
	u32* counts = ctx->counts;
	const u32 C = ctx->cfg.max_contacts, S = ctx->stride;
	k_cache_lookup<<<GRID(C), NB_BLOCK, 0, st>>>(ctx->fin.tags, ctx->fin.features, ctx->cache_tags, ctx->cache_features, ctx->cache_data, ctx->impulses, counts);
	k_culled_flags<<<GRID(C), NB_BLOCK, 0, st>>>(ctx->cache_tags, ctx->sleeping, flags, counts);
	ctx->launches += 2;
	nb_scan<1>(L, flags, offs, S, counts + CNT_CACHE, 0, block_sums, counts + CNT_CULLED);
	k_culled_scatter<<<GRID(C), NB_BLOCK, 0, st>>>(flags, offs, ctx->cache_tags, ctx->cache_features, ctx->cache_data,
		ctx->culled_tags, ctx->culled_features, ctx->culled_data, counts);
	++ctx->launches;
	CK(cudaGetLastError());
	return NB_OK;
}

static int read_sort(nb_context* ctx, void* stream) {
	Launch L = mk_launch(ctx, stream);
	cudaStream_t st = L.stream;
	u32* counts = ctx->counts;
	const u32 C = ctx->cfg.max_contacts;
	// order contacts by tag: stable sort on the feature word, then on the pair word (nudge.cpp:4024-4044)
	int cur;
	if (ctx->contacts_internal && 2 * ctx->tagbits + 16 <= 64) {
		const u32 spread = (ctx->tagbits >= 3 && 2 * ctx->tagbits + 17 <= 64) ? 1u : 0u;
		k_tag_keys_packed<<<GRID(C), NB_BLOCK, 0, st>>>(ctx->fin.tags, ctx->fin.features, ctx->sb.keys[0], ctx->sb.vals[0], ctx->tagbits, spread, counts); ++ctx->launches;
		cur = nb_radix_sort(L, ctx->sb, counts + CNT_CONTACTS, 0, (int)(2 * ctx->tagbits + 16 + spread), true, 0);
	}
	else {  // contacts supplied through nb_upload_contacts: arbitrary feature words
		k_tag_keys_feature<<<GRID(C), NB_BLOCK, 0, st>>>(ctx->fin.features, ctx->sb.keys[0], ctx->sb.vals[0], counts); ++ctx->launches;
		cur = nb_radix_sort(L, ctx->sb, counts + CNT_CONTACTS, 0, 32, true, 0);
		k_tag_keys_pair<<<GRID(C), NB_BLOCK, 0, st>>>(ctx->fin.tags, ctx->sb.vals[cur], ctx->sb.keys[cur], ctx->tagbits, counts); ++ctx->launches;
		cur = nb_radix_sort(L, ctx->sb, counts + CNT_CONTACTS, 0, (int)(2 * ctx->tagbits), true, cur);
	}
	k_copy_u32<<<GRID(C), NB_BLOCK, 0, st>>>(ctx->sb.vals[cur], ctx->sorted, counts + CNT_CONTACTS);
	++ctx->launches;
	CK(cudaGetLastError());
	return NB_OK;
}

int nb_read_cached_impulses(nb_context* ctx, void* stream) {
	NB_RANGE("nb_read_cached_impulses");
	int r = read_sort(ctx, stream); if (r) return r;
	return read_lookup(ctx, (cudaStream_t)stream, ctx->flags, ctx->offs, ctx->block_sums);
}

int nb_write_cached_impulses(nb_context* ctx, void* stream) {
	NB_RANGE("nb_write_cached_impulses");
	const u32 C = ctx->cfg.max_contacts;
	k_cache_merge<<<GRID(C), NB_BLOCK, 0, (cudaStream_t)stream>>>(ctx->sorted, ctx->fin.tags, ctx->fin.features, ctx->impulses,
		ctx->culled_tags, ctx->culled_features, ctx->culled_data, ctx->cache_tags, ctx->cache_features, ctx->cache_data, ctx->counts);
	++ctx->launches;
	CK(cudaGetLastError());
	return NB_OK;
}

// ---------------- setup + solve ----------------
static void timing_begin(nb_context* ctx, cudaStream_t st) {
	if (!ctx->timing || ctx->capturing || ctx->tev_n >= 64) return;
	if (!ctx->tev_made) { for (int i = 0; i < 64; ++i) { cudaEventCreate(&ctx->tev[0][i]); cudaEventCreate(&ctx->tev[1][i]); } ctx->tev_made = true; }
	cudaEventRecord(ctx->tev[0][ctx->tev_n], st);
}
static void timing_end(nb_context* ctx, cudaStream_t st) {
	if (!ctx->timing || ctx->capturing || ctx->tev_n >= 64) return;
	cudaEventRecord(ctx->tev[1][ctx->tev_n++], st);
}

// throughput mode: warm start and sweeps as Jacobi passes (k_jacobi_sweep + k_jacobi_apply per pass), nb_jacobi.cuh
static int launch_solve_jacobi(nb_context* ctx, int mode, u32 sweeps, cudaStream_t st) {
	Rows R = ctx->rows;
	const u32 B = ctx->B;
	k_mw_in<<<GRID(B), NB_BLOCK, 0, st>>>(B, ctx->mom, ctx->mw);
	++ctx->launches;
	// two tiles per CTA in flight once the body arrays (64 B per body: velocities + accumulators) take a large share of L2, else more CTAs
	const int stages = ctx->jacobi_stages == 1 || ctx->jacobi_stages == 2 ? ctx->jacobi_stages : (B > 600000u ? 2 : 1);
	if (mode == 0 || mode == 2) {
		if (stages == 1) k_jacobi_sweep<true, 1><<<ctx->jacobi_blocks1, NJ_TILE, sizeof(JacobiSmem<1>), st>>>(R, ctx->impulses, ctx->mw, ctx->jd, ctx->counts);
		else k_jacobi_sweep<true, 2><<<ctx->jacobi_blocks2, NJ_TILE, sizeof(JacobiSmem<2>), st>>>(R, ctx->impulses, ctx->mw, ctx->jd, ctx->counts);
		k_jacobi_apply<<<GRID(B), NB_BLOCK, 0, st>>>(B, ctx->mw, ctx->jd, ctx->jcnt);
		ctx->launches += 2;
	}
	if (mode != 0)
		for (u32 w = 0; w < sweeps; ++w) {
			timing_begin(ctx, st);
			if (stages == 1) k_jacobi_sweep<false, 1><<<ctx->jacobi_blocks1, NJ_TILE, sizeof(JacobiSmem<1>), st>>>(R, ctx->impulses, ctx->mw, ctx->jd, ctx->counts);
			else k_jacobi_sweep<false, 2><<<ctx->jacobi_blocks2, NJ_TILE, sizeof(JacobiSmem<2>), st>>>(R, ctx->impulses, ctx->mw, ctx->jd, ctx->counts);
			timing_end(ctx, st);
			k_jacobi_apply<<<GRID(B), NB_BLOCK, 0, st>>>(B, ctx->mw, ctx->jd, ctx->jcnt);
			ctx->launches += 2;
		}
	k_mw_out<<<GRID(B), NB_BLOCK, 0, st>>>(B, ctx->mom, ctx->mw, mode ? 1 : 0);
	++ctx->launches;
	return NB_OK;
}

// the exact-order solver kernel alone, on a working copy `mw` that the caller has filled (k_mw_in or the sharded step's fused pull)
static int launch_solve_core(nb_context* ctx, int mode, u32 sweeps, cudaStream_t st) {
	Rows R = ctx->rows;
	const float4* impulses = ctx->impulses;
	float4* mw = ctx->mw;
	u32* counts = ctx->counts;
	u32 backoff = ctx->solve_backoff_ns;
	void* args[] = { &R, &impulses, &mw, &mode, &sweeps, &backoff, &counts };
	if (mode) timing_begin(ctx, st);
	if (ctx->coop_launch && (!ctx->capturing || ctx->graph_coop)) CK(cudaLaunchCooperativeKernel(ctx->solve_wide ? (void*)k_solve<true> : (void*)k_solve<false>, dim3(ctx->coop_blocks_solve), dim3(NB_BLOCK), args, 0, st));
	else if (ctx->solve_wide) k_solve<true><<<ctx->coop_blocks_solve, NB_BLOCK, 0, st>>>(R, impulses, mw, mode, sweeps, backoff, counts);
	else k_solve<false><<<ctx->coop_blocks_solve, NB_BLOCK, 0, st>>>(R, impulses, mw, mode, sweeps, backoff, counts);
	if (mode) timing_end(ctx, st);
	++ctx->launches;
	return NB_OK;
}

static int launch_solve(nb_context* ctx, int mode, u32 sweeps, cudaStream_t st) {
	if (ctx->solver_mode == NB_SOLVER_THROUGHPUT) return launch_solve_jacobi(ctx, mode, sweeps, st);
	const u32 B = ctx->B;
	k_mw_in<<<GRID(B), NB_BLOCK, 0, st>>>(B, ctx->mom, ctx->mw);
	int r = launch_solve_core(ctx, mode, sweeps, st); if (r) return r;
	k_mw_out<<<GRID(B), NB_BLOCK, 0, st>>>(B, ctx->mom, ctx->mw, mode ? 1 : 0);
	ctx->launches += 2;
	return NB_OK;
}

int nb_setup_contact_constraints(nb_context* ctx, void* stream) {
	NB_RANGE("nb_setup_contact_constraints");
	JOIN_UPLOADS();
	Launch L = mk_launch(ctx, stream);
	cudaStream_t st = L.stream;
	u32* counts = ctx->counts;
	const u32 C = ctx->cfg.max_contacts, S = ctx->stride, B = ctx->B;
	k_inertia<<<GRID(B), NB_BLOCK, 0, st>>>(B, ctx->xf, ctx->props, ctx->inertia, ctx->mom);
	if (ctx->solver_mode == NB_SOLVER_THROUGHPUT) {
		// no batch schedule, no per-body chains: slots in tag order, per-body contact counts for the mass split, split rows
		CK(cudaMemsetAsync(ctx->rows.contact, 0xff, sizeof(u32) * ctx->cstride, st));
		CK(cudaMemsetAsync(ctx->jcnt, 0, sizeof(u32) * B, st));
		k_jacobi_prepare<<<GRID(C), NB_BLOCK, 0, st>>>(ctx->sorted, ctx->fin.bodies, ctx->jcnt, ctx->rows, ctx->cstride, counts);
		k_build_rows<true><<<GRID(ctx->cstride), NB_BLOCK, 0, st>>>(ctx->fin.data, ctx->fin.bodies, ctx->xf, ctx->inertia, ctx->mom, ctx->rows, counts, ctx->jcnt);
		ctx->launches += 3;
		if (!ctx->defer_warm_start) {
			if (ctx->join_before_solve) { ctx->join_before_solve = false; CK(cudaStreamWaitEvent(st, ctx->ev_join, 0)); }   // the warm start reads the looked-up impulses
			int r = launch_solve(ctx, 0, 1, st); if (r) return r; if (ctx->urow_n && (r = launch_user_rows(ctx, 1, st))) return r;
		}
		CK(cudaGetLastError());
		return NB_OK;
	}
	k_sched_prep<<<GRID(C), NB_BLOCK, 0, st>>>(ctx->sorted, ctx->fin.bodies, ctx->cab, ctx->back, counts);
	k_schedule<<<16, 32, 0, st>>>(ctx->cab, ctx->back, ctx->slot_of, ctx->slot_done, ctx->slot_left, ctx->slots_per_bucket,
		ctx->flags, ctx->left_count, ctx->sched_spill_ent, ctx->sched_spill_uid, ctx->sched_spill_cap, counts);
	ctx->launches += 3;
	nb_scan<1>(L, ctx->flags, ctx->offs, S, counts + CNT_CONTACTS, 0, ctx->block_sums, counts + CNT_FULL_BATCHES);
	// key layout of the per-body chain sort: (body | batch).  Sides on the static world become dummies spread over the unused part
	// of the body field (an extra bit if less than a quarter of it is free), so no sort bucket collects them all.
	u32 chain_bodybits = bits_for(std::max(B, 2u));
	if (((u64)1 << chain_bodybits) - B < ((u64)1 << chain_bodybits) / 4) ++chain_bodybits;
	const u32 dummy_span = (u32)std::min<u64>(((u64)1 << chain_bodybits) - B, 0x7fffffffu);
	CK(cudaMemsetAsync(ctx->rows.contact, 0xff, sizeof(u32) * ctx->cstride, st));
	k_batch_index<<<GRID(C), NB_BLOCK, 0, st>>>(ctx->sorted, ctx->fin.bodies, ctx->slot_of, ctx->slot_done, ctx->slot_left, ctx->slots_per_bucket,
		ctx->offs, ctx->left_count, ctx->batch_of, ctx->slot_idx, ctx->rows.contact, ctx->cstride, ctx->sb.keys[0], ctx->sb.vals[0], ctx->batchbits, B, dummy_span, counts);
	++ctx->launches;
	if (ctx->rows_on_side) CK(cudaEventRecord(ctx->ev_fork2, st));   // slots are final here
	int cur = nb_radix_sort(L, ctx->sb, counts + CNT_ENTRIES, 0, (int)(chain_bodybits + ctx->batchbits), true, 0);
	if (ctx->zero_chain_len) CK(cudaMemsetAsync(ctx->chain_len, 0, sizeof(u32) * B, st));
	k_chain_heads<<<GRID(2 * C), NB_BLOCK, 0, st>>>(ctx->sb.keys[cur], ctx->batchbits, B, ctx->chain_start, ctx->chain_len, counts); ++ctx->launches;
	k_waits<<<GRID(2 * C), NB_BLOCK, 0, st>>>(ctx->sb.keys[cur], ctx->sb.vals[cur], ctx->batchbits, B, ctx->slot_idx, ctx->chain_start, ctx->chain_len, ctx->rows.wait, ctx->cstride, counts);
	// the rows only need the slot of every contact (k_batch_index), not the chains: inside nb_step they are built on the second stream
	// while the chain sort runs (rows_stream != st; joined before the solver)
	cudaStream_t rows_stream = ctx->rows_on_side ? ctx->side : st;
	if (ctx->rows_on_side) CK(cudaStreamWaitEvent(ctx->side, ctx->ev_fork2, 0));
	k_build_rows<false><<<GRID(ctx->cstride), NB_BLOCK, 0, rows_stream>>>(ctx->fin.data, ctx->fin.bodies, ctx->xf, ctx->inertia, ctx->mom, ctx->rows, counts, nullptr);
	if (ctx->rows_on_side) { CK(cudaEventRecord(ctx->ev_join2, ctx->side)); CK(cudaStreamWaitEvent(st, ctx->ev_join2, 0)); }
	ctx->launches += 2;
	if (!ctx->defer_warm_start) {  // warm start (nudge.cpp:4563-4632), then the user rows' accumulated impulses
		if (ctx->join_before_solve) { ctx->join_before_solve = false; CK(cudaStreamWaitEvent(st, ctx->ev_join, 0)); }
		int r = launch_solve(ctx, 0, 1, st); if (r) return r;
		if (ctx->urow_n && (r = launch_user_rows(ctx, 1, st))) return r;
	}
	CK(cudaGetLastError());
	return NB_OK;
}

int nb_apply_impulses(nb_context* ctx, uint32_t sweeps, void* stream) {
	NB_RANGE("nb_apply_impulses");
	JOIN_UPLOADS();
	if (!sweeps) return NB_OK;
	if (ctx->urow_n && !ctx->defer_warm_start) {   // user rows run after EVERY sweep (example/main.cpp:314-317): one sweep per solver launch
		for (uint32_t w = 0; w < sweeps; ++w) {
			int r = launch_solve(ctx, 1, 1, (cudaStream_t)stream); if (r) return r;
			if ((r = launch_user_rows(ctx, 0, (cudaStream_t)stream))) return r;
		}
		return NB_OK;
	}
	int r = launch_solve(ctx, ctx->defer_warm_start ? 2 : 1, sweeps, (cudaStream_t)stream); if (r) return r;
	ctx->defer_warm_start = false;
	CK(cudaGetLastError());
	return NB_OK;
}

int nb_update_cached_impulses(nb_context* ctx, void* stream) {
	NB_RANGE("nb_update_cached_impulses");
	k_update_impulses<<<GRID(ctx->cstride), NB_BLOCK, 0, (cudaStream_t)stream>>>(ctx->rows, ctx->impulses, ctx->counts);
	++ctx->launches;
	CK(cudaGetLastError());
	return NB_OK;
}

int nb_advance(nb_context* ctx, float time_step, void* stream) {
	NB_RANGE("nb_advance");
	JOIN_UPLOADS();
	k_advance<<<GRID(ctx->B), NB_BLOCK, 0, (cudaStream_t)stream>>>(ctx->active_idx, ctx->xf, ctx->mom, ctx->idle, time_step, ctx->counts);
	++ctx->launches;
	CK(cudaGetLastError());
	return NB_OK;
}

static int step_body(nb_context* ctx, float time_step, uint32_t iterations, float gravity, float damping, void* stream) {
	int r;
	if ((r = nb_collide(ctx, stream))) return r;
	if ((r = nb_apply_gravity_damping(ctx, time_step, gravity, damping, stream))) return r;
	const bool fork = ctx->overlap && stream != nullptr && !ctx->debug;
	cudaStream_t st = (cudaStream_t)stream;
	if (fork) {
		// branch A on the second stream: cache lookup + culled entries (needs the contacts and the sorted sleeping pairs, not the tag order);
		// it joins before the solver's warm start reads the impulses.  Own scan scratch: the scheduler uses the main one meanwhile.
		CK(cudaEventRecord(ctx->ev_fork, st)); CK(cudaStreamWaitEvent(ctx->side, ctx->ev_fork, 0));
		if ((r = read_lookup(ctx, ctx->side, ctx->flags2, ctx->offs2, ctx->block_sums2))) return r;
		CK(cudaEventRecord(ctx->ev_join, ctx->side));
		if ((r = read_sort(ctx, stream))) return r;
	}
	else if ((r = nb_read_cached_impulses(ctx, stream))) return r;
	ctx->defer_warm_start = iterations > 0 && !ctx->urow_n;  // warm start + sweeps in one solver launch (same arithmetic, same order); not with user rows between the sweeps
	ctx->rows_on_side = fork && ctx->solver_mode == NB_SOLVER_PARITY;   // branch B: constraint rows while the chain sort runs
	ctx->join_before_solve = fork;
	r = nb_setup_contact_constraints(ctx, stream);
	ctx->rows_on_side = false;
	if (!r && ctx->join_before_solve) { ctx->join_before_solve = false; CK(cudaStreamWaitEvent(st, ctx->ev_join, 0)); }   // (setup joins itself when it runs the warm start)
	if (!r) r = nb_apply_impulses(ctx, iterations, stream);
	ctx->defer_warm_start = false; ctx->join_before_solve = false;
	if (r) return r;
	if ((r = nb_update_cached_impulses(ctx, stream))) return r;
	if ((r = nb_write_cached_impulses(ctx, stream))) return r;
	return nb_advance(ctx, time_step, stream);
}

// One sub-step (example/main.cpp:274-328).  On a capturable stream the ~75 launches are recorded once into a CUDA graph and
// replayed; every count the kernels need lives in device memory, so the graph only depends on the parameters and the scene
// shape held in StepKey.  NB_GRAPH=0, the legacy default stream or debug mode use plain launches.
int nb_step(nb_context* ctx, float time_step, uint32_t iterations, float gravity, float damping, void* stream) {
	NB_RANGE("nb_step");
	cudaStream_t st = (cudaStream_t)stream;
	if (!ctx->graph_enabled || st == nullptr || st == cudaStreamLegacy || st == cudaStreamPerThread || ctx->debug)
		return step_body(ctx, time_step, iterations, gravity, damping, stream);
	nb_context::StepKey key;
	memset(&key, 0, sizeof(key));  // padding bytes included: the key is compared with memcmp
	key.stream = st; key.ts = time_step; key.gravity = gravity; key.damping = damping; key.iterations = iterations;
	key.B = ctx->B; key.nboxes = ctx->nboxes; key.nspheres = ctx->nspheres; key.nconn = ctx->nconn; key.tagbits = ctx->tagbits; key.kbits = ctx->kbits; key.debug = ctx->debug; key.solver_mode = ctx->solver_mode; key.urow_version = ctx->urow_version;
	if (!ctx->graph_exec || memcmp(&key, &ctx->graph_key, sizeof(key)) != 0) {
		if (ctx->graph_exec) { cudaGraphExecDestroy(ctx->graph_exec); ctx->graph_exec = nullptr; }
		// Attempt 1 keeps the cooperative-launch attribute on the grid-synchronising kernel nodes (k_sort_coop's software grid barriers,
		// k_solve's spin waits): the driver then guarantees co-residency at replay, also with other work on the device.  If this
		// driver refuses cooperative nodes in a capture, attempt 2 records them as ordinary nodes (correct on an otherwise idle device:
		// their grids are sized from the occupancy calculator), and if that fails too the step stays on plain launches.
		for (int attempt = ctx->graph_coop ? 0 : 1; attempt < 2 && !ctx->graph_exec; ++attempt) {
			const unsigned long long before = ctx->launches;
			const int coop = ctx->sb.coop_launch, gcoop = ctx->graph_coop;
			if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); break; }
			ctx->capturing = true; ctx->capture_joined = false;
			if (attempt == 1) { ctx->sb.coop_launch = 0; ctx->graph_coop = 0; }
			int r = step_body(ctx, time_step, iterations, gravity, damping, stream);
			ctx->capturing = false; ctx->sb.coop_launch = coop; ctx->graph_coop = gcoop;
			cudaGraph_t graph = nullptr;
			cudaError_t e = cudaStreamEndCapture(st, &graph);
			if (r == NB_OK && e == cudaSuccess && graph) e = cudaGraphInstantiate(&ctx->graph_exec, graph, 0);
			if (graph) cudaGraphDestroy(graph);
			ctx->graph_launches = ctx->launches - before;
			ctx->launches = before;
			if (r != NB_OK || e != cudaSuccess || !ctx->graph_exec) { cudaGetLastError(); ctx->graph_exec = nullptr; if (attempt == 0) ctx->graph_coop = 0; }
			else ctx->graph_is_coop = attempt == 0;
		}
		if (!ctx->graph_exec) {  // capture refused: stay on plain launches
			ctx->graph_enabled = 0;
			return step_body(ctx, time_step, iterations, gravity, damping, stream);
		}
		ctx->graph_key = key;
	}
	CK(cudaGraphLaunch(ctx->graph_exec, st));
	ctx->upload_pending = false;   // the graph's event-wait node has ordered this replay after the side copy
	ctx->launches += ctx->graph_launches;
	ctx->contacts_internal = true;
	return NB_OK;
}

// ---------------- streams for hosts that do not link the CUDA runtime themselves ----------------
void* nb_stream_create(nb_context* ctx) {
	cudaStream_t s = nullptr;
	if (cudaSetDevice(ctx->cfg.device) != cudaSuccess || cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess) { ctx->error = "cudaStreamCreate failed"; return nullptr; }
	return (void*)s;
}
void nb_stream_destroy(nb_context* ctx, void* stream) { (void)ctx; if (stream) { cudaStreamSynchronize((cudaStream_t)stream); cudaStreamDestroy((cudaStream_t)stream); } }
int nb_stream_synchronize(nb_context* ctx, void* stream) { CK(cudaStreamSynchronize((cudaStream_t)stream)); return NB_OK; }

// ---------------- solver mode and kernel timing ----------------
int nb_set_solver_mode(nb_context* ctx, int mode) {
	if (mode != NB_SOLVER_PARITY && mode != NB_SOLVER_THROUGHPUT) { ctx->error = "unknown solver mode"; return NB_ERR_ARGUMENT; }
	ctx->solver_mode = mode;
	return NB_OK;
}
int nb_get_solver_mode(const nb_context* ctx) { return ctx->solver_mode; }

// CUDA events around every launch of the dominant solver kernel (k_solve in parity mode, k_jacobi_sweep in throughput mode) while
// enabled; plain launches only (the stage calls, or nb_step with NB_GRAPH=0).  nb_debug_timing synchronises the stream and returns
// the number of timed launches and their summed duration, then clears the list.
int nb_debug_timing_enable(nb_context* ctx, int on) { ctx->timing = on; ctx->tev_n = 0; return NB_OK; }
int nb_debug_timing(nb_context* ctx, uint32_t* launches, float* total_ms, void* stream) {
	CK(cudaStreamSynchronize((cudaStream_t)stream));
	float sum = 0.0f;
	for (int i = 0; i < ctx->tev_n; ++i) { float ms = 0.0f; CK(cudaEventElapsedTime(&ms, ctx->tev[0][i], ctx->tev[1][i])); sum += ms; }
	if (launches) *launches = (uint32_t)ctx->tev_n;
	if (total_ms) *total_ms = sum;
	ctx->tev_n = 0;
	return NB_OK;
}

// ---------------- parity-test introspection ----------------
int nb_debug_read(nb_context* ctx, const char* name, void* dst, size_t max_bytes, size_t* bytes, void* stream) {
	u32 c[CNT__COUNT];
	int r = get_counts(ctx, c, stream); if (r) return r;
	const u32 K = ctx->nboxes + ctx->nspheres;
	struct Entry { const char* name; const void* ptr; size_t bytes; };
	const Entry table[] = {
		{ "counts", ctx->counts, sizeof(u32) * CNT__COUNT },
		{ "order", ctx->order, sizeof(u32) * K },
		{ "aabb_min", ctx->aabb_min, sizeof(float4) * K },
		{ "aabb_max", ctx->aabb_max, sizeof(float4) * K },
		{ "world_xf", ctx->world_xf, sizeof(nb_transform) * K },
		{ "pair_keys", ctx->pair_keys_debug, sizeof(u64) * (ctx->pair_keys_debug ? c[CNT_PAIRS] : 0) },
		{ "live", ctx->live, sizeof(uint2) * c[CNT_LIVE_TOTAL] },
		{ "sorted", ctx->sorted, sizeof(u32) * c[CNT_CONTACTS] },
		{ "impulses", ctx->impulses, sizeof(float4) * c[CNT_CONTACTS] },
		{ "culled_tags", ctx->culled_tags, sizeof(u64) * c[CNT_CULLED] },
		{ "culled_features", ctx->culled_features, sizeof(u32) * c[CNT_CULLED] },
		{ "culled_data", ctx->culled_data, sizeof(float4) * c[CNT_CULLED] },
		{ "batch_of", ctx->batch_of, sizeof(u32) * c[CNT_CONTACTS] },
		{ "slot_idx", ctx->slot_idx, sizeof(u32) * c[CNT_CONTACTS] },
		{ "row_contact", ctx->rows.contact, sizeof(u32) * 8 * c[CNT_BATCHES] },
		{ "row_a", ctx->rows.a, sizeof(u32) * 8 * c[CNT_BATCHES] },
		{ "row_b", ctx->rows.b, sizeof(u32) * 8 * c[CNT_BATCHES] },
		{ "row_wait", ctx->rows.wait, sizeof(uint2) * 2 * (size_t)ctx->cstride },
		{ "row_planes", ctx->rows.plane, sizeof(float) * (size_t)ROW_PLANES * ctx->cstride },
		{ "row_states", ctx->rows.state, sizeof(float) * 3 * (size_t)ctx->cstride },
		{ "inertia", ctx->inertia, sizeof(float4) * 2 * ctx->B },
		{ "row_planes_all", ctx->rows.plane, sizeof(float) * (size_t)ROW_PLANES_TOTAL * ctx->cstride },
		{ "body_contacts", ctx->jcnt, sizeof(u32) * ctx->B },
		{ "query_world_xf", ctx->q.world_xf, sizeof(nb_transform) * ctx->q.K },
	};
	if (!strcmp(name, "row_stride")) { if (max_bytes < 4) return NB_ERR_ARGUMENT; *(u32*)dst = ctx->cstride; if (bytes) *bytes = 4; return NB_OK; }
	if (!strcmp(name, "graph_coop")) { if (max_bytes < 4) return NB_ERR_ARGUMENT; *(u32*)dst = ctx->graph_exec ? (ctx->graph_is_coop ? 2u : 1u) : 0u; if (bytes) *bytes = 4; return NB_OK; }
	if (!strcmp(name, "kbits")) { if (max_bytes < 4) return NB_ERR_ARGUMENT; *(u32*)dst = ctx->kbits; if (bytes) *bytes = 4; return NB_OK; }
	for (size_t i = 0; i < sizeof(table) / sizeof(table[0]); ++i)
		if (!strcmp(name, table[i].name)) {
			if (bytes) *bytes = table[i].bytes;
			if (!dst) return NB_OK;
			if (table[i].bytes > max_bytes) { ctx->error = "debug buffer too small"; return NB_ERR_CAPACITY; }
			CK(cudaMemcpyAsync(dst, table[i].ptr, table[i].bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
			CK(cudaStreamSynchronize((cudaStream_t)stream));
			return NB_OK;
		}
	ctx->error = std::string("unknown debug buffer ") + name;
	return NB_ERR_ARGUMENT;
}

// Keeps a copy of the sorted broadphase pair list for nb_debug_read("pair_keys") (one extra copy kernel per collide).
int nb_debug_enable(nb_context* ctx, int on) {
	if (on && !ctx->pair_keys_debug) ALLOC(ctx->pair_keys_debug, ctx->cfg.max_pairs);
	ctx->debug = on;
	return NB_OK;
}

// Runs the device radix sort / scan on host data (unit tests of the primitives).
int nb_debug_sort(nb_context* ctx, uint64_t* keys, uint32_t* vals, uint32_t n, int begin_bit, int end_bit) {
	if (n > ctx->sort_cap) { ctx->error = "too many keys"; return NB_ERR_CAPACITY; }
	Launch L = mk_launch(ctx, nullptr);
	CK(cudaMemcpy(ctx->sb.keys[0], keys, (size_t)n * 8, cudaMemcpyHostToDevice));
	if (vals) CK(cudaMemcpy(ctx->sb.vals[0], vals, (size_t)n * 4, cudaMemcpyHostToDevice));
	CK(cudaMemcpy(ctx->counts + CNT_SCRATCH1, &n, 4, cudaMemcpyHostToDevice));
	int cur = nb_radix_sort(L, ctx->sb, ctx->counts + CNT_SCRATCH1, begin_bit, end_bit, vals != nullptr, 0);
	CK(cudaMemcpy(keys, ctx->sb.keys[cur], (size_t)n * 8, cudaMemcpyDeviceToHost));
	if (vals) CK(cudaMemcpy(vals, ctx->sb.vals[cur], (size_t)n * 4, cudaMemcpyDeviceToHost));
	return NB_OK;
}
int nb_debug_scan(nb_context* ctx, uint32_t* data, uint32_t n, uint32_t* total) {
	if (n > ctx->stride) { ctx->error = "too many values"; return NB_ERR_CAPACITY; }
	Launch L = mk_launch(ctx, nullptr);
	CK(cudaMemcpy(ctx->flags, data, (size_t)n * 4, cudaMemcpyHostToDevice));
	CK(cudaMemcpy(ctx->counts + CNT_SCRATCH1, &n, 4, cudaMemcpyHostToDevice));
	nb_scan<1>(L, ctx->flags, ctx->offs, ctx->stride, ctx->counts + CNT_SCRATCH1, 0, ctx->block_sums, ctx->counts + CNT_SCRATCH0);
	CK(cudaMemcpy(data, ctx->offs, (size_t)n * 4, cudaMemcpyDeviceToHost));
	CK(cudaMemcpy(total, ctx->counts + CNT_SCRATCH0, 4, cudaMemcpyDeviceToHost));
	return NB_OK;
}

int nb_debug_rcp(nb_context* ctx, const float* x, float* y, uint32_t n, int rsq) {
	float* dx = (float*)ctx->sb.keys[0]; float* dy = (float*)ctx->sb.keys[1];
	if ((size_t)n * 4 > (size_t)ctx->sort_cap * 8) { ctx->error = "too many probes"; return NB_ERR_CAPACITY; }
	CK(cudaMemcpy(dx, x, (size_t)n * 4, cudaMemcpyHostToDevice));
	k_debug_rcp<<<GRID(n), NB_BLOCK>>>(dx, dy, n, rsq); ++ctx->launches;
	CK(cudaMemcpy(y, dy, (size_t)n * 4, cudaMemcpyDeviceToHost));
	return NB_OK;
}

}

#include "nb_shard_api.cuh"
#include "nb_state_api.cuh"
#include "nb_rows_api.cuh"
#include "nb_render_api.cuh"
#include "nb_query_api.cuh"
