// tw_voxel_post.cu - voxel post-processing on the device (SURVEY.md 8f row N3): the steps of voxel_model::build after the density fill
// (src/voxels.cpp:1496-1530): determine_voxels_outside (:571-604), remove_unconnected_outside / remove_interior_holes (:606-610, :729-868) and the marching
// cubes of add_triangles_for_voxel (:485-566) for the whole grid in create_block order (:1077-1108). Layout: index z + (x + y*nx)*nz (src/voxels.h:141-144).
//   outside_kernel      one thread per voxel, streaming (4 B read + 1 B written per voxel)
//   flood fills         breadth-first frontier expansion: a voxel is claimed by whoever first sets its ANCHORED bit (atomicOr on the 32-bit word that holds
//                       its flag byte), so it enters the next frontier exactly once; the SET of reached voxels is what the reference's depth-first stack
//                       reaches, the visiting order is irrelevant. 8 expansion launches per host check of the frontier size.
//   mc_kernel<EMIT>     1024 consecutive voxels per block = 1024 cubes in the reference's (y, x, z) order; every thread builds its cube's <= 5 triangles,
//                       a block scan of the per-cube counts plus the scanned block totals give every triangle its slot, i.e. the output is in the
//                       reference's emission order without atomics (pass 1: counts only; pass 2: write).
// All fp32 arithmetic is the reference's (separate multiply and add: the TU is compiled with -fmad=false), std::min/max argument order kept.
#include "tw_internal.h"
#include <vector>

namespace {

constexpr float VOX_TOLERANCE = 1.0E-12f; // TOLERANCE, src/3DWorld.h:50

__device__ __forceinline__ float smin(float a, float b) {return (b < a) ? b : a;} // std::min
__device__ __forceinline__ float smax(float a, float b) {return (a < b) ? b : a;} // std::max

__global__ void outside_kernel(const float *__restrict__ vals, tw_voxel_post_params P, const unsigned *__restrict__ zix_xy, unsigned char *__restrict__ outside, size_t n) {
	size_t const stride = (size_t)gridDim.x*blockDim.x;
	for (size_t i = (size_t)blockIdx.x*blockDim.x + threadIdx.x; i < n; i += stride) {
		unsigned const z = (unsigned)(i % P.nz);
		size_t const xy = i / P.nz;
		unsigned const x = (unsigned)(xy % P.nx), y = (unsigned)(xy / P.nx);
		bool const on_edge = (P.make_closed_surface && ((x == 0 || x == P.nx-1) || (y == 0 || y == P.ny-1) || (z == 0 || z == P.nz-1)));
		float const val = __ldg(vals + i);
		unsigned char ival = on_edge ? (unsigned char)TW_VOX_ON_EDGE : (unsigned char)((val == P.isolevel) ? 1 : (((val < P.isolevel) != (P.invert != 0)) ? 1 : 0)); // val_is_outside
		if (zix_xy && z < __ldg(zix_xy + (size_t)y*P.nx + x)) {ival |= TW_VOX_UNDER_MESH;}
		outside[i] = ival;
	}
}

// ---- flood fill ----
__device__ __forceinline__ bool claim(unsigned char *outside, size_t ix, unsigned char fill_val, unsigned char bit) { // outside[ix] == fill_val -> |= bit, true for exactly one caller
	if (*(volatile unsigned char *)(outside + ix) != fill_val) return false;
	unsigned *word = (unsigned *)(outside + (ix & ~(size_t)3));
	unsigned const shift = (unsigned)(ix & 3)*8u;
	unsigned const old = atomicOr(word, (unsigned)bit << shift);
	return (((old >> shift) & 0xffu) == fill_val);
}
// seeds of remove_unconnected_outside_range (src/voxels.cpp:768-805); mode 0: voxels under the mesh (outside == UNDER_MESH), 1: scene-edge columns (outside != 1),
// 2: top plane of remove_interior_holes (outside != 0, :835-842)
__global__ void seed_kernel(unsigned char *outside, tw_voxel_post_params P, int mode, unsigned *frontier, unsigned *count, size_t n) {
	size_t const stride = (size_t)gridDim.x*blockDim.x;
	for (size_t i = (size_t)blockIdx.x*blockDim.x + threadIdx.x; i < n; i += stride) {
		unsigned char const o = outside[i];
		bool seed = false;
		if (mode == 0) {seed = (o == TW_VOX_UNDER_MESH);}
		else {
			unsigned const z = (unsigned)(i % P.nz);
			size_t const xy = i / P.nz;
			unsigned const x = (unsigned)(xy % P.nx), y = (unsigned)(xy / P.nx);
			if (mode == 1) {seed = ((x == 0 || x + 1 == P.nx || y == 0 || y + 1 == P.ny) && o != 1 && !(o & TW_VOX_ANCHORED));}
			else           {seed = (z == P.nz - 1 && o != 0);}
		}
		if (seed) { // flag bytes of one word may be seeded by different threads: set the bit atomically
			unsigned *word = (unsigned *)(outside + (i & ~(size_t)3));
			atomicOr(word, (unsigned)TW_VOX_ANCHORED << ((unsigned)(i & 3)*8u));
			frontier[atomicAdd(count, 1u)] = (unsigned)i;
		}
	}
}
__global__ void seed_centre_kernel(unsigned char *outside, tw_voxel_post_params P, unsigned *frontier, unsigned *count) { // :769-776
	size_t const ix = (P.nz/2) + ((size_t)(P.nx/2) + (size_t)(P.ny/2)*P.nx)*P.nz;
	outside[ix] |= TW_VOX_ANCHORED;
	frontier[atomicAdd(count, 1u)] = (unsigned)ix;
}
// flood_fill_range + FLOOD_FILL_INNER (src/voxels.cpp:729-757) for one frontier generation
__global__ void flood_expand_kernel(unsigned char *outside, unsigned nx, unsigned ny, unsigned nz, const unsigned *__restrict__ fin, const unsigned *__restrict__ n_in,
	unsigned *__restrict__ fout, unsigned *__restrict__ n_out, unsigned char fill_val, unsigned char bit)
{
	unsigned const n = *n_in, nxnz = nx*nz;
	for (unsigned i = blockIdx.x*blockDim.x + threadIdx.x; i < n; i += gridDim.x*blockDim.x) {
		unsigned const cur = fin[i];
		unsigned const y = cur/nxnz, cur_xz = cur - y*nxnz, x = cur_xz/nz, z = cur_xz - x*nz;
#define TW_FF(pos, max_range, step) \
		if (pos >= 1)            {unsigned const ix = cur - step; if (claim(outside, ix, fill_val, bit)) {fout[atomicAdd(n_out, 1u)] = ix;}} \
		if (pos + 1 < max_range) {unsigned const ix = cur + step; if (claim(outside, ix, fill_val, bit)) {fout[atomicAdd(n_out, 1u)] = ix;}}
		TW_FF(x, nx, nz)
		TW_FF(y, ny, nxnz)
		TW_FF(z, nz, 1u)
#undef TW_FF
	}
}
// :808-826 (pass 0) and :847-857 (pass 1)
__global__ void flood_finish_kernel(float *__restrict__ vals, unsigned char *__restrict__ outside, float isolevel, int invert, int pass, unsigned long long *changed, size_t n) {
	size_t const stride = (size_t)gridDim.x*blockDim.x;
	unsigned long long c = 0;
	for (size_t i = (size_t)blockIdx.x*blockDim.x + threadIdx.x; i < n; i += stride) {
		unsigned char const o = outside[i];
		if (pass == 0) {
			if (o > 1) {outside[i] = o & (unsigned char)~TW_VOX_ANCHORED;}
			else if (o != 1) {outside[i] = 1; vals[i] = isolevel - (invert ? -VOX_TOLERANCE : VOX_TOLERANCE); ++c;} // make_voxel_outside, :861-864
		}
		else {
			if (o & TW_VOX_ANCHORED) {outside[i] = o & (unsigned char)~TW_VOX_ANCHORED;}
			else if (o == 1) {outside[i] = 0; vals[i] = isolevel + (invert ? -VOX_TOLERANCE : VOX_TOLERANCE); ++c;} // make_voxel_inside, :865-868
		}
	}
	for (int o = 16; o > 0; o >>= 1) {c += __shfl_xor_sync(0xffffffffu, c, o);}
	if ((threadIdx.x & 31) == 0 && c) {atomicAdd(changed, c);}
}

// ---- marching cubes ----
struct McTables {const unsigned *edge_table; const int *tri_table; const unsigned *edge_to_vals;};
constexpr int MC_BLOCK = 1024;

__device__ __forceinline__ void interpolate_pt(float isolevel, const float *pt1, const float *pt2, float val1, float val2, float *pt) { // src/voxels.cpp:485-493
	if (fabsf(isolevel - val1) < VOX_TOLERANCE) {pt[0] = pt1[0]; pt[1] = pt1[1]; pt[2] = pt1[2]; return;}
	if (fabsf(isolevel - val2) < VOX_TOLERANCE) {pt[0] = pt2[0]; pt[1] = pt2[1]; pt[2] = pt2[2]; return;}
	if (fabsf(val1     - val2) < VOX_TOLERANCE) {pt[0] = pt1[0]; pt[1] = pt1[1]; pt[2] = pt1[2]; return;}
	float const mu = smax(0.0f, smin(1.0f, __fdiv_rn(isolevel - val1, val2 - val1))); // CLIP_TO_01
#pragma unroll
	for (int i = 0; i < 3; ++i) {pt[i] = pt1[i] + mu*(pt2[i] - pt1[i]);}
}

// add_triangles_for_voxel(x, y, z) at lod 0 (src/voxels.cpp:495-566): returns the number of valid triangles, written to tri[k][9] when EMIT
template<bool EMIT>
__device__ unsigned cube_triangles(const float *__restrict__ vals, const unsigned char *__restrict__ outside, const tw_voxel_post_params &P, const McTables &T,
	unsigned x, unsigned y, unsigned z, float (*tri)[9])
{
	unsigned const nx = P.nx, ny = P.ny, nz = P.nz;
	unsigned const x2 = min(x + 1, nx - 1), y2 = min(y + 1, ny - 1), z2 = min(z + 1, nz - 1);
	if (x2 <= x || y2 <= y || z2 <= z) return 0; // invalid (empty) range
	unsigned const xv[2] = {x, x2}, yv[2] = {y, y2}, zv[2] = {z, z2};
	unsigned cix = 0;
	bool all_under_mesh = (P.skip_under_mesh != 0);
#pragma unroll
	for (unsigned yhi = 0; yhi < 2; ++yhi) {
#pragma unroll
		for (unsigned xhi = 0; xhi < 2; ++xhi) {
			size_t const ix = z + ((size_t)xv[xhi] + (size_t)yv[yhi]*nx)*nz;
			if (all_under_mesh) {all_under_mesh = ((__ldg(outside + ix) & TW_VOX_UNDER_MESH) != 0);}
#pragma unroll
			for (unsigned zhi = 0; zhi < 2; ++zhi) {if (__ldg(outside + ix + zv[zhi] - z) & 7) {cix |= 1u << ((xhi ^ yhi) + 2*yhi + 4*zhi);}} // outside or on edge
		}
	}
	if (all_under_mesh) return 0;
	unsigned const edge_val = __ldg(T.edge_table + cix);
	if (edge_val == 0) return 0; // no polygons
	const int *t = T.tri_table + 16*cix;
	float const cube[3][2] = {{(float)x*P.vsz[0] + P.lo_pos[0], (float)x2*P.vsz[0] + P.lo_pos[0]}, {(float)y*P.vsz[1] + P.lo_pos[1], (float)y2*P.vsz[1] + P.lo_pos[1]},
	                          {(float)z*P.vsz[2] + P.lo_pos[2], (float)z2*P.vsz[2] + P.lo_pos[2]}}; // get_xv / get_yv / get_zv
	float vlist[12][3];
	for (unsigned i = 0; i < 12; ++i) {
		if (!(edge_val & (1u << i))) continue;
		float v2[2], pts[2][3];
#pragma unroll
		for (unsigned d = 0; d < 2; ++d) {
			unsigned const e = __ldg(T.edge_to_vals + 2*i + d), yhi = (e & 2) >> 1, xhi = yhi ^ (e & 1), zhi = e >> 2;
			size_t const ix = zv[zhi] + ((size_t)xv[xhi] + (size_t)yv[yhi]*nx)*nz;
			v2[d] = ((__ldg(outside + ix) & 7) == TW_VOX_ON_EDGE) ? P.isolevel : __ldg(vals + ix);
			pts[d][0] = cube[0][xhi]; pts[d][1] = cube[1][yhi]; pts[d][2] = cube[2][zhi];
		}
		interpolate_pt(P.isolevel, pts[0], pts[1], v2[0], v2[1], vlist[i]);
	}
	unsigned count = 0;
	for (unsigned i = 0; i < 15; i += 3) {
		int const t0 = __ldg(t + i);
		if (t0 < 0) break;
		const float *p0 = vlist[t0], *p1 = vlist[__ldg(t + i + 1)], *p2 = vlist[__ldg(t + i + 2)];
		float const a0 = p1[0] - p0[0], a1 = p1[1] - p0[1], a2 = p1[2] - p0[2], b0 = p2[0] - p1[0], b1 = p2[1] - p1[1], b2 = p2[2] - p1[2]; // get_normal: cross(v2 - v1, v3 - v2)
		float const cx = a1*b2 - a2*b1, cy = a2*b0 - a0*b2, cz = a0*b1 - a1*b0;
		if (cx == 0.0f && cy == 0.0f && cz == 0.0f) continue; // normal == zero_vector: invalid triangle (:550)
		if (EMIT) {
#pragma unroll
			for (int k = 0; k < 3; ++k) {tri[count][k] = p0[k]; tri[count][3 + k] = p1[k]; tri[count][6 + k] = p2[k];}
		}
		++count;
	}
	return count;
}

template<bool EMIT>
__global__ void __launch_bounds__(MC_BLOCK)
mc_kernel(const float *__restrict__ vals, const unsigned char *__restrict__ outside, tw_voxel_post_params P, McTables T, size_t n, unsigned *__restrict__ block_sums,
	const unsigned long long *__restrict__ block_offsets, float *__restrict__ tris, unsigned long long capacity)
{
	__shared__ unsigned warp_sums[MC_BLOCK/32];
	size_t const i = (size_t)blockIdx.x*MC_BLOCK + threadIdx.x;
	float tri[5][9];
	unsigned cnt = 0;
	if (i < n) {
		unsigned const z = (unsigned)(i % P.nz);
		size_t const xy = i / P.nz;
		cnt = cube_triangles<EMIT>(vals, outside, P, T, (unsigned)(xy % P.nx), (unsigned)(xy / P.nx), z, tri);
	}
	// exclusive scan of cnt over the block (cube order == thread order)
	unsigned const lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	unsigned incl = cnt;
	for (int o = 1; o < 32; o <<= 1) {unsigned const v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= (unsigned)o) incl += v;}
	if (lane == 31) {warp_sums[warp] = incl;}
	__syncthreads();
	if (warp == 0) {
		unsigned w = warp_sums[lane], wi = w;
		for (int o = 1; o < 32; o <<= 1) {unsigned const v = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= (unsigned)o) wi += v;}
		warp_sums[lane] = wi - w; // exclusive
		if (!EMIT && lane == 31) {block_sums[blockIdx.x] = wi;}
	}
	__syncthreads();
	if (EMIT && cnt) {
		unsigned long long const base = block_offsets[blockIdx.x] + warp_sums[warp] + (incl - cnt);
		for (unsigned k = 0; k < cnt; ++k) {
			unsigned long long const slot = base + k;
			if (slot < capacity) {float *o = tris + 9*slot; for (int c = 0; c < 9; ++c) {o[c] = tri[k][c];}}
		}
	}
}
// exclusive scan of the block totals into 64-bit offsets (one block; nblocks is ~1e5 for a 512^3 grid); total[0] = grand total
__global__ void __launch_bounds__(1024)
scan_blocks_kernel(const unsigned *__restrict__ sums, unsigned nblocks, unsigned long long *__restrict__ offsets, unsigned long long *__restrict__ total) {
	__shared__ unsigned long long warp_sums[32];
	__shared__ unsigned long long carry;
	if (threadIdx.x == 0) {carry = 0;}
	__syncthreads();
	unsigned const lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	for (unsigned base = 0; base < nblocks; base += 1024) {
		unsigned const i = base + threadIdx.x;
		unsigned long long const v = (i < nblocks) ? sums[i] : 0ull;
		unsigned long long incl = v;
		for (int o = 1; o < 32; o <<= 1) {unsigned long long const u = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= (unsigned)o) incl += u;}
		if (lane == 31) {warp_sums[warp] = incl;}
		__syncthreads();
		if (warp == 0) {
			unsigned long long w = warp_sums[lane], wi = w;
			for (int o = 1; o < 32; o <<= 1) {unsigned long long const u = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= (unsigned)o) wi += u;}
			warp_sums[lane] = wi - w;
		}
		__syncthreads();
		unsigned long long const excl = carry + warp_sums[warp] + (incl - v);
		if (i < nblocks) {offsets[i] = excl;}
		__syncthreads();
		if (threadIdx.x == 1023) {carry = excl + v;}
		__syncthreads();
	}
	if (threadIdx.x == 0) {*total = carry;}
}

int validate(tw_ctx *ctx, const tw_voxel_post_params *vp) {
	if (!vp || vp->nx == 0 || vp->ny == 0 || vp->nz == 0) return tw_set_error(ctx, TW_ERR_ARG, "empty voxel grid");
	if ((unsigned long long)vp->nx*vp->ny*vp->nz >= 0xffffffffull) return tw_set_error(ctx, TW_ERR_ARG, "voxel grids are indexed with 32 bits, as in the reference (src/voxels.h:141)");
	return TW_OK;
}
unsigned stream_grid(size_t n) {size_t const b = (n + 255)/256; return (unsigned)(b < 148u*16u ? (b ? b : 1) : 148u*16u);}

} // namespace

extern "C" int tw_voxel_outside(tw_ctx *ctx, const float *vals, const tw_voxel_post_params *vp, const uint32_t *zix_xy, uint8_t *outside) {
	int rc = tw_enter(ctx); if (rc) return rc;
	if (!vals || !outside) return tw_set_error(ctx, TW_ERR_ARG, "null argument");
	rc = validate(ctx, vp); if (rc) return rc;
	size_t const n = (size_t)vp->nx*vp->ny*vp->nz;
	const float *d_v; uint8_t *d_o; const uint32_t *d_z;
	tw_stage st(ctx);
	st.in(&d_v, vals, n*sizeof(float));
	st.out(&d_o, outside, n);
	st.in(&d_z, zix_xy, (size_t)vp->nx*vp->ny*sizeof(uint32_t));
	rc = st.commit(); if (rc) return rc;
	outside_kernel<<<stream_grid(n), 256, 0, ctx->stream>>>(d_v, *vp, d_z, d_o, n);
	TW_LAUNCH_CHECK(ctx);
	return st.finish();
}

// one flood fill: frontier buffers f[0], f[1] (n + 16 entries each), counters cnt[0], cnt[1]; the seeds are already in f[0] / cnt[0]
static int run_flood(tw_ctx *ctx, unsigned char *d_o, const tw_voxel_post_params *vp, unsigned *f[2], unsigned *cnt, unsigned char fill_val, unsigned char bit) {
	int cur = 0;
	for (;;) {
		for (int k = 0; k < 8; ++k) {
			TW_CUDA(ctx, cudaMemsetAsync(cnt + (cur ^ 1), 0, sizeof(unsigned), ctx->stream));
			flood_expand_kernel<<<148*4, 256, 0, ctx->stream>>>(d_o, vp->nx, vp->ny, vp->nz, f[cur], cnt + cur, f[cur ^ 1], cnt + (cur ^ 1), fill_val, bit);
			TW_LAUNCH_CHECK(ctx);
			cur ^= 1;
		}
		unsigned h = 0;
		TW_CUDA(ctx, cudaMemcpyAsync(&h, cnt + cur, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
		TW_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
		if (h == 0) return TW_OK;
	}
}

extern "C" int tw_voxel_remove_unconnected(tw_ctx *ctx, float *vals, uint8_t *outside, const tw_voxel_post_params *vp, uint64_t *changed) {
	int rc = tw_enter(ctx); if (rc) return rc;
	if (!vals || !outside) return tw_set_error(ctx, TW_ERR_ARG, "null argument");
	rc = validate(ctx, vp); if (rc) return rc;
	if (changed) *changed = 0;
	if (vp->remove_unconnected <= 0) return TW_OK;
	size_t const n = (size_t)vp->nx*vp->ny*vp->nz;
	float *d_v; uint8_t *d_o; unsigned *f[2], *cnt;
	tw_stage st(ctx);
	st.inout(&d_v, vals, n*sizeof(float));
	st.inout(&d_o, outside, n, 4); // + 4: claim() sets flag bytes with atomics on the 32-bit word that holds them
	st.temp(&f[0], (n + 16)*sizeof(unsigned));
	st.temp(&f[1], (n + 16)*sizeof(unsigned));
	st.temp(&cnt, 128); // cnt[0], cnt[1]; the changed counter at byte 64
	rc = st.commit(); if (rc) return rc;
	if ((size_t)d_o & 3) return tw_set_error(ctx, TW_ERR_ARG, "outside must be 4-byte aligned (flag bytes are claimed with 32-bit atomics)"); // only a device buffer can be
	unsigned long long *d_changed = (unsigned long long *)((char *)cnt + 64);
	TW_CUDA(ctx, cudaMemsetAsync(cnt, 0, 128, ctx->stream));
	// remove_unconnected_outside_range(keep_at_edge, 0, 0, nx, ny): anchors, fill of the inside voxels, verdict
	if (vp->centre_seed) {seed_centre_kernel<<<1, 1, 0, ctx->stream>>>(d_o, *vp, f[0], cnt);}
	else {seed_kernel<<<stream_grid(n), 256, 0, ctx->stream>>>(d_o, *vp, 0, f[0], cnt, n);}
	TW_LAUNCH_CHECK(ctx);
	if (vp->keep_at_edge) {seed_kernel<<<stream_grid(n), 256, 0, ctx->stream>>>(d_o, *vp, 1, f[0], cnt, n); TW_LAUNCH_CHECK(ctx);}
	rc = run_flood(ctx, d_o, vp, f, cnt, 0, TW_VOX_ANCHORED); if (rc) return rc;
	flood_finish_kernel<<<stream_grid(n), 256, 0, ctx->stream>>>(d_v, d_o, vp->isolevel, vp->invert, 0, d_changed, n);
	TW_LAUNCH_CHECK(ctx);
	if (vp->remove_unconnected > 2) { // remove_interior_holes
		TW_CUDA(ctx, cudaMemsetAsync(cnt, 0, 2*sizeof(unsigned), ctx->stream));
		seed_kernel<<<stream_grid(n), 256, 0, ctx->stream>>>(d_o, *vp, 2, f[0], cnt, n);
		TW_LAUNCH_CHECK(ctx);
		unsigned h = 0;
		TW_CUDA(ctx, cudaMemcpyAsync(&h, cnt, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
		TW_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
		if (h) { // "can't find empty space for the seed, bail out" otherwise (:844)
			rc = run_flood(ctx, d_o, vp, f, cnt, 1, TW_VOX_ANCHORED); if (rc) return rc;
			flood_finish_kernel<<<stream_grid(n), 256, 0, ctx->stream>>>(d_v, d_o, vp->isolevel, vp->invert, 1, d_changed, n);
			TW_LAUNCH_CHECK(ctx);
		}
	}
	unsigned long long hc = 0;
	TW_CUDA(ctx, cudaMemcpyAsync(&hc, d_changed, sizeof(hc), cudaMemcpyDeviceToHost, ctx->stream));
	rc = st.finish(); if (rc) return rc;
	if (changed) *changed = hc;
	return TW_OK;
}

extern "C" int tw_voxel_triangles(tw_ctx *ctx, const float *vals, const uint8_t *outside, const tw_voxel_post_params *vp, const uint32_t *edge_table256,
                                  const int32_t *tri_table256x16, const uint32_t *edge_to_vals12x2, float *tris, uint64_t capacity, uint64_t *ntris)
{
	int rc = tw_enter(ctx); if (rc) return rc;
	if (!vals || !outside || !edge_table256 || !tri_table256x16 || !edge_to_vals12x2 || !ntris || (capacity && !tris)) return tw_set_error(ctx, TW_ERR_ARG, "null argument");
	rc = validate(ctx, vp); if (rc) return rc;
	size_t const n = (size_t)vp->nx*vp->ny*vp->nz;
	unsigned const nblocks = (unsigned)((n + MC_BLOCK - 1)/MC_BLOCK);
	const float *d_v; const uint8_t *d_o; McTables T; unsigned *d_sums; unsigned long long *d_offsets, *d_total;
	tw_stage st(ctx);
	st.in(&d_v, vals, n*sizeof(float));
	st.in(&d_o, outside, n);
	st.in(&T.edge_table, edge_table256, 256*sizeof(uint32_t));
	st.in(&T.tri_table, tri_table256x16, 256*16*sizeof(int32_t));
	st.in(&T.edge_to_vals, edge_to_vals12x2, 12*2*sizeof(uint32_t));
	st.temp(&d_sums, (size_t)nblocks*sizeof(unsigned));
	st.temp(&d_offsets, (size_t)nblocks*sizeof(unsigned long long));
	st.temp(&d_total, sizeof(unsigned long long));
	rc = st.commit(); if (rc) return rc;
	mc_kernel<false><<<nblocks, MC_BLOCK, 0, ctx->stream>>>(d_v, d_o, *vp, T, n, d_sums, nullptr, nullptr, 0);
	TW_LAUNCH_CHECK(ctx);
	scan_blocks_kernel<<<1, 1024, 0, ctx->stream>>>(d_sums, nblocks, d_offsets, d_total);
	TW_LAUNCH_CHECK(ctx);
	unsigned long long total = 0;
	TW_CUDA(ctx, cudaMemcpyAsync(&total, d_total, sizeof(total), cudaMemcpyDeviceToHost, ctx->stream));
	TW_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	*ntris = total;
	if (capacity == 0 || total == 0) return TW_OK;
	uint64_t const nw = (total < capacity) ? total : capacity;
	float *d_t = tris;
	bool const host_t = tw_stage::is_host(tris);
	if (host_t) {rc = tw_reserve(ctx, 1, (size_t)nw*9*sizeof(float)); if (rc) return rc; d_t = (float *)ctx->d_scratch[1];}
	mc_kernel<true><<<nblocks, MC_BLOCK, 0, ctx->stream>>>(d_v, d_o, *vp, T, n, nullptr, d_offsets, d_t, nw);
	TW_LAUNCH_CHECK(ctx);
	if (host_t) {TW_CUDA(ctx, cudaMemcpyAsync(tris, d_t, (size_t)nw*9*sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));}
	TW_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	return TW_OK;
}
