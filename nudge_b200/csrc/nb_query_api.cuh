// nudge_b200 — ray casts against the device-resident scene (DESIGN.md §8.5; no reference counterpart).
//
// nb_build_query_tree snapshots the scene into buffers of its own with the collision stage's kernels (k_collider_world -> k_morton ->
// nb_radix_sort -> k_leaves -> k_build_level), so the snapshot's world transforms are bit for bit what nb_collide computes, and nothing the
// step reads or counts is written.  k_raycast walks the implicit 8-ary AABB tree, one thread per ray, nearest child first, and decides
// every hit with the exact float32 shape tests below.  The tree only prunes: its boxes are widened (conservative culling, see
// NB_QUERY_PAD) and a node is skipped only when its entry t is strictly greater than the best t so far, so with the tie rule (equal t:
// smaller collider index) the result does not depend on tree shape, ray order or launch configuration.
// Algorithmic bytes: 32 in (nb_ray) + 32 out (nb_ray_hit) per ray, plus node reads (32 B per tested child, 48 B per exactly tested
// collider); the tree is about 1.14 K x 32 B and stays L2-resident up to millions of colliders.
// Included at the end of nb_api.cu.
#pragma once

// Relative widening of the culling boxes.  The exact tests work in the collider's frame; the float AABB (|R| s summed in float) and the
// float slab test of a node carry rounding errors of a few ulps of the coordinates involved, and a grazing sphere hit (disc near 0) can
// land up to eps |m|^2 / (2 r) outside the sphere's box.  Every leaf box grows by PAD (max |coordinate| + 1) and every ray pads the node
// slabs by PAD (max |origin| + 1), which covers these errors with a wide margin (for spheres while |origin - centre| < ~1000 r).
#define NB_QUERY_PAD (1.0f / 8192.0f)
#define NB_QUERY_BIG 1e30f   // |1/d| clamp of the node test: a zero direction component gives no NaN

// Morton-ordered collider records for the traversal (3 float4 per leaf: position + body bits, rotation, size or radius + collider
// index bits), and the widened leaf boxes.
__global__ void __launch_bounds__(NB_BLOCK) k_query_leaves(u32 K, u32 nboxes, const u32* order, const nb_transform* world_xf, const nb_box_collider* box_data,
		const nb_sphere_collider* sph_data, float4* leaf_min, float4* leaf_max, float4* rec) {
	for (u32 pos = blockIdx.x * blockDim.x + threadIdx.x; pos < K; pos += gridDim.x * blockDim.x) {
		const u32 i = order[pos];
		const xform w = ld_xform(world_xf, i);
		float4 s;
		if (i < nboxes) s = reinterpret_cast<const float4*>(box_data)[i];
		else { const float r = sph_data[i - nboxes].radius; s = make_float4(r, r, r, 0.0f); }
		s.w = asf(i);
		rec[3 * (size_t)pos] = w.p; rec[3 * (size_t)pos + 1] = w.q; rec[3 * (size_t)pos + 2] = s;
		float4 lo = leaf_min[pos], hi = leaf_max[pos];
		const float m = fmaxf(fmaxf(fmaxf(fabsf(lo.x), fabsf(lo.y)), fmaxf(fabsf(lo.z), fabsf(hi.x))), fmaxf(fabsf(hi.y), fabsf(hi.z)));
		const float pad = NB_QUERY_PAD * (m + 1.0f);
		lo.x -= pad; lo.y -= pad; lo.z -= pad; hi.x += pad; hi.y += pad; hi.z += pad;
		leaf_min[pos] = lo; leaf_max[pos] = hi;
	}
}

// ---- exact shape tests (DESIGN.md §8.5 fixes the operation order; -fmad=false keeps every * and + a separate rounding) ----
// Box: ray into the box frame with the conjugate rotation, slabs against the half extents.  Returns false on a miss.
NB_DEV bool q_box(f3 o, f3 d, float4 p, float4 q, float4 s, float& t, f3& n) {
	quat qc; qc.v = mk3(nb_neg(q.x), nb_neg(q.y), nb_neg(q.z)); qc.s = q.w;
	const f3 ol = qrot(qc, sub3(o, mk3(p.x, p.y, p.z)));
	const f3 dl = qrot(qc, d);
	const float oa[3] = { ol.x, ol.y, ol.z }, da[3] = { dl.x, dl.y, dl.z }, sa[3] = { s.x, s.y, s.z };
	float tnear = -INFINITY, tfar = INFINITY;
	int axis = -1;
	#pragma unroll
	for (int k = 0; k < 3; ++k) {
		if (da[k] == 0.0f) { if (!(fabsf(oa[k]) <= sa[k])) return false; }   // parallel to the slab: inside iff |o| <= s (no 0 * inf)
		else {
			const float enter = ((da[k] > 0.0f ? nb_neg(sa[k]) : sa[k]) - oa[k]) / da[k];
			const float leave = ((da[k] > 0.0f ? sa[k] : nb_neg(sa[k])) - oa[k]) / da[k];
			if (enter > tnear) { tnear = enter; axis = k; }   // strict: tied slabs keep the lowest axis
			if (leave < tfar) tfar = leave;
		}
	}
	if (!(tnear <= tfar) || !(tfar >= 0.0f)) return false;
	if (tnear > 0.0f) {
		const float sg = da[axis] > 0.0f ? -1.0f : 1.0f;
		t = tnear;
		n = qrot(mkq(q), mk3(axis == 0 ? sg : 0.0f, axis == 1 ? sg : 0.0f, axis == 2 ? sg : 0.0f));
	}
	else { t = 0.0f; n = mk3(0.0f, 0.0f, 0.0f); }   // origin inside (boundary included)
	return true;
}

NB_DEV bool q_sphere(f3 o, f3 d, float4 p, float r, float& t, f3& n) {
	const f3 c = mk3(p.x, p.y, p.z);
	const f3 m = sub3(o, c);
	const float a = dot3(d, d), b = dot3(m, d), cc = dot3(m, m) - r * r;
	if (cc <= 0.0f) { t = 0.0f; n = mk3(0.0f, 0.0f, 0.0f); return true; }   // origin inside (boundary included)
	const float disc = b * b - a * cc;
	if (!(disc >= 0.0f) || !(a > 0.0f)) return false;
	const float tt = (nb_neg(b) - sqrtf(disc)) / a;
	if (!(tt >= 0.0f)) return false;
	t = tt;
	n = mk3(((o.x + tt * d.x) - c.x) / r, ((o.y + tt * d.y) - c.y) / r, ((o.z + tt * d.z) - c.z) / r);
	return true;
}

// Padded slab test of a culling box: entry t in `tn`; true if the box may hold a hit at t <= best.
struct QRay { float ox, oy, oz, ix, iy, iz, px, py, pz; };
NB_DEV bool q_node(const QRay& R, float4 lo, float4 hi, float best, float& tn) {
	const float ax = (lo.x - R.ox) * R.ix, bx = (hi.x - R.ox) * R.ix;
	const float ay = (lo.y - R.oy) * R.iy, by = (hi.y - R.oy) * R.iy;
	const float az = (lo.z - R.oz) * R.iz, bz = (hi.z - R.oz) * R.iz;
	tn = fmaxf(fmaxf(fminf(ax, bx) - R.px, fminf(ay, by) - R.py), fminf(az, bz) - R.pz);
	const float tf = fminf(fminf(fmaxf(ax, bx) + R.px, fmaxf(ay, by) + R.py), fmaxf(az, bz) + R.pz);
	return tn <= tf && tf >= 0.0f && tn <= best;
}

// One thread per ray.  Stack: per level a queue of up to 8 child slots (3 bits each, nearest first, count in bits 24..27); the node
// being visited at every level follows from the current block's first child (`base`), since an implicit tree's parent is index / 8.
__global__ void __launch_bounds__(NB_BLOCK) k_raycast(Tree T, u32 nboxes, const float4* __restrict__ rec, const u32* __restrict__ tags, const nb_ray* __restrict__ rays,
		nb_ray_hit* __restrict__ hits, u32 n) {
	for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
		const float4 r0 = reinterpret_cast<const float4*>(rays)[2 * (size_t)i], r1 = reinterpret_cast<const float4*>(rays)[2 * (size_t)i + 1];
		const f3 o = mk3(r0.x, r0.y, r0.z), d = mk3(r1.x, r1.y, r1.z);
		const u32 ignore = asu(r1.w);
		float best = r0.w;
		u32 best_c = NB_NO_BODY, best_b = NB_NO_BODY;
		f3 best_n = mk3(0.0f, 0.0f, 0.0f);
		QRay R;
		R.ox = o.x; R.oy = o.y; R.oz = o.z;
		R.ix = fminf(fmaxf(1.0f / d.x, -NB_QUERY_BIG), NB_QUERY_BIG);
		R.iy = fminf(fmaxf(1.0f / d.y, -NB_QUERY_BIG), NB_QUERY_BIG);
		R.iz = fminf(fmaxf(1.0f / d.z, -NB_QUERY_BIG), NB_QUERY_BIG);
		{
			const float pad = NB_QUERY_PAD * (fmaxf(fmaxf(fabsf(o.x), fabsf(o.y)), fabsf(o.z)) + 1.0f);
			R.px = pad * fabsf(R.ix); R.py = pad * fabsf(R.iy); R.pz = pad * fabsf(R.iz);
		}
		const int top = T.levels - 1;
		u32 queue[NB_MAX_LEVELS];
		int level = top;                     // level of the block of children tested next
		u32 base = 0, cnt = top >= 0 ? T.n[top] : 0;   // the top level (<= 8 nodes) is the block of a virtual root
		while (top >= 0) {
			const float4* mn = T.mn[level];
			const float4* mx = T.mx[level];
			if (level == 0) {
				#pragma unroll
				for (u32 c = 0; c < 8; ++c) {
					float tn;
					if (c < cnt && q_node(R, mn[base + c], mx[base + c], best, tn)) {
						const size_t leaf = 3 * (size_t)(base + c);
						const float4 p = rec[leaf];
						if (asu(p.w) == ignore) continue;
						const float4 q = rec[leaf + 1], s = rec[leaf + 2];
						const u32 ci = asu(s.w);
						float t; f3 nn;
						if (!(ci < nboxes ? q_box(o, d, p, q, s, t, nn) : q_sphere(o, d, p, s.x, t, nn))) continue;
						if (t < best || (t == best && ci < best_c)) { best = t; best_c = ci; best_b = asu(p.w); best_n = nn; }
					}
				}
			}
			else {
				float tn[8];
				u32 mask = 0;
				#pragma unroll
				for (u32 c = 0; c < 8; ++c) {
					tn[c] = INFINITY;
					if (c < cnt && q_node(R, mn[base + c], mx[base + c], best, tn[c])) mask |= 1u << c;
				}
				u32 qv = 0, qn = 0;
				#pragma unroll
				for (int k = 0; k < 8; ++k) {   // selection order by entry t
					if (!mask) break;
					float bt = INFINITY; u32 bc = __ffs(mask) - 1;
					#pragma unroll
					for (u32 c = 0; c < 8; ++c) if (((mask >> c) & 1u) && tn[c] < bt) { bt = tn[c]; bc = c; }
					qv |= bc << (3 * qn); ++qn; mask &= ~(1u << bc);
				}
				queue[level] = qv | (qn << 24);
			}
			// next block: the nearest queued child at the lowest level that still has one, re-tested against the best t so far (the queue
			// is in entry-t order, so the first child that fails ends its whole queue)
			bool found = false;
			u32 node = 0;
			int l = level == 0 ? 1 : level;
			for (; l <= top; ++l) {
				const u32 bl = (base >> (3 * (l - level))) & ~7u;
				u32 qv = queue[l];
				while (qv >> 24) {
					const u32 c = qv & 7u;
					qv = ((qv & 0xffffffu) >> 3) | (((qv >> 24) - 1) << 24);
					float tn;
					if (q_node(R, T.mn[l][bl + c], T.mx[l][bl + c], best, tn)) { node = bl + c; found = true; break; }
					qv = 0;
				}
				queue[l] = qv;
				if (found) break;
			}
			if (!found) break;
			level = l - 1; base = node * 8; cnt = min(8u, T.n[level] - base);
		}
		const u32 tag = best_c != NB_NO_BODY ? tags[best_c] : NB_NO_BODY;
		float4* h = reinterpret_cast<float4*>(hits) + 2 * (size_t)i;
		h[0] = make_float4(best, asf(best_c), asf(best_b), asf(tag));
		h[1] = make_float4(best_n.x, best_n.y, best_n.z, 0.0f);
	}
}

static void dev_free(nb_context* ctx, void* p) {
	if (!p) return;
	cudaFree(p);
	ctx->allocs.erase(std::remove(ctx->allocs.begin(), ctx->allocs.end(), p), ctx->allocs.end());
}

// The snapshot's buffers, sized from the configured capacities (like ctx->instances): allocated by the first nb_build_query_tree, so a
// context that never casts a ray pays nothing.
static int query_alloc(nb_context* ctx) {
	nb_context::Query& q = ctx->q;
	if (q.counts) return NB_OK;
	const u32 K = std::max(1u, ctx->cfg.max_boxes + ctx->cfg.max_spheres);
	size_t tree_nodes = K; { u32 n = K; while (n > 8) { n = (n + 7) / 8; tree_nodes += n; } }
	ALLOC(q.world_xf, K); ALLOC(q.aabb_min, K); ALLOC(q.aabb_max, K); ALLOC(q.col_tag, K); ALLOC(q.col_body, K);
	ALLOC(q.order, K); ALLOC(q.rank, K); ALLOC(q.mkeys, K); ALLOC(q.leaf, 3 * (size_t)K);
	ALLOC(q.tree_min, tree_nodes + 8); ALLOC(q.tree_max, tree_nodes + 8);
	for (int i = 0; i < 2; ++i) { ALLOC(q.sb.keys[i], K); ALLOC(q.sb.vals[i], K); }
	ALLOC(q.sb.hist, 256 * NB_SORT_GRID); ALLOC(q.sb.block_sums, 8 * NB_SCAN_GRID);
	ALLOC(q.keybits, 2);
	ALLOC(q.counts, CNT__COUNT);   // last: it marks the set as allocated
	q.sb.bar = q.counts + CNT_BAR0;
	CK(cudaDeviceSynchronize());   // the zero fills (grid-barrier counters among them) are done before any stream uses the buffers
	return NB_OK;
}

extern "C" {

int nb_build_query_tree(nb_context* ctx, void* stream) {
	NB_RANGE("nb_build_query_tree");
	int r = query_alloc(ctx); if (r) return r;
	nb_context::Query& q = ctx->q;
	Launch L = mk_launch(ctx, stream);
	cudaStream_t st = L.stream;
	const u32 K = ctx->B ? ctx->nboxes + ctx->nspheres : 0;
	Tree& T = q.T;
	T.levels = 0;
	if (K) {
		size_t off = 0; u32 n = K; int l = 0;
		while (true) {
			if (l == NB_MAX_LEVELS) { ctx->error = "too many colliders for the query tree (8^9)"; return NB_ERR_CAPACITY; }
			T.mn[l] = q.tree_min + off; T.mx[l] = q.tree_max + off; T.n[l] = n; off += n; ++l;
			if (n <= 8) break;
			n = (n + 7) / 8;
		}
		T.levels = l;
		q.sb.coop_blocks = ctx->sb.coop_blocks; q.sb.coop_launch = ctx->sb.coop_launch;
		k_reset_collide<<<1, 32, 0, st>>>(q.counts, K, q.keybits);
		k_collider_world<<<GRID(K), NB_BLOCK, 0, st>>>(ctx->nboxes, ctx->nspheres, ctx->xf, ctx->box_xf, ctx->box_data, ctx->box_tags,
			ctx->sph_xf, ctx->sph_data, ctx->sph_tags, q.world_xf, q.aabb_min, q.aabb_max, q.col_tag, q.col_body, q.counts);
		k_morton<<<GRID(K), NB_BLOCK, 0, st>>>(K, q.aabb_min, q.aabb_max, q.counts, q.sb.keys[0], q.sb.vals[0], q.keybits);
		ctx->launches += 3;
		const int cur = nb_radix_sort(L, q.sb, q.counts + CNT_SCRATCH1, 0, 48, true, 0, 0, 0, q.keybits);
		k_leaves<<<GRID(K), NB_BLOCK, 0, st>>>(K, q.sb.vals[cur], q.sb.keys[cur], q.aabb_min, q.aabb_max, q.order, q.rank, (float4*)T.mn[0], (float4*)T.mx[0], q.mkeys);
		// the snapshot's sizes travel in the leaf records: a later nb_upload_colliders with the same counts does not reach the rays
		k_query_leaves<<<GRID(K), NB_BLOCK, 0, st>>>(K, ctx->nboxes, q.order, q.world_xf, ctx->box_data, ctx->sph_data, (float4*)T.mn[0], (float4*)T.mx[0], q.leaf);
		ctx->launches += 2;
		for (int l = 1; l < T.levels; ++l) {
			k_build_level<<<GRID(T.n[l]), NB_BLOCK, 0, st>>>(T.mn[l - 1], T.mx[l - 1], T.n[l - 1], (float4*)T.mn[l], (float4*)T.mx[l], T.n[l]);
			++ctx->launches;
		}
	}
	CK(cudaGetLastError());
	q.built = true; q.nboxes = ctx->nboxes; q.nspheres = ctx->nspheres; q.K = K;
	return NB_OK;
}

int nb_raycast(nb_context* ctx, const nb_ray* rays, nb_ray_hit* hits, uint32_t n, int io_is_device, void* stream) {
	NB_RANGE("nb_raycast");
	nb_context::Query& q = ctx->q;
	cudaStream_t st = (cudaStream_t)stream;
	if (!q.built) { ctx->error = "nb_raycast: no query tree (call nb_build_query_tree first)"; return NB_ERR_ARGUMENT; }
	if (q.nboxes != ctx->nboxes || q.nspheres != ctx->nspheres) { ctx->error = "nb_raycast: the collider counts changed since nb_build_query_tree"; return NB_ERR_ARGUMENT; }
	if (!n) return NB_OK;
	if (!rays || !hits) { ctx->error = "nb_raycast: null rays or hits"; return NB_ERR_ARGUMENT; }
	const nb_ray* dr = rays;
	nb_ray_hit* dh = hits;
	if (!io_is_device) {
		if (q.io_cap < n) {
			dev_free(ctx, q.rays); dev_free(ctx, q.hits); q.rays = nullptr; q.hits = nullptr; q.io_cap = 0;
			u32 cap = 1024; while (cap < n && cap < 0x80000000u) cap *= 2;
			cap = std::max(cap, n);
			ALLOC(q.rays, cap); ALLOC(q.hits, cap);
			q.io_cap = cap;
		}
		H2D(q.rays, rays, n, nb_ray);
		dr = q.rays; dh = q.hits;
	}
	k_raycast<<<(n + NB_BLOCK - 1) / NB_BLOCK, NB_BLOCK, 0, st>>>(q.T, q.nboxes, q.leaf, q.col_tag, dr, dh, n);
	++ctx->launches;
	CK(cudaGetLastError());
	if (!io_is_device) {
		D2H(hits, q.hits, n, nb_ray_hit);
		CK(cudaStreamSynchronize(st));
	}
	return NB_OK;
}

}  // extern "C"
