// tw_shadows.cu - mesh shadows of tiles (SURVEY.md 8f row N4): calc_mesh_shadows / mesh_shadow_gen (src/visibility.cpp:411-517) with the neighbour chaining of
// tile_t::calc_shadows_for_light (src/tiled_mesh.cpp:664-692). The reference traces 2*ysize rays from the tile's x edge and 2*xsize from its y edge (half-cell
// spacing) along the light's shadow direction, each a Bresenham walk that carries the running shadow height; rays are independent except for what they leave behind:
//   smask |= MESH_SHADOW            order-free: atomicOr on the 32-bit word that holds the flag byte
//   sh_out_x / sh_out_y[...] = z    last writer wins in the reference's sequential order (run_x rays by y, then run_y rays by x): a 64-bit atomicMax on
//                                   (ray number + 1) << 32 | float bits picks exactly that writer; a second small kernel unpacks the keys
// One thread per ray, all tiles of a dependency wave in one launch (a tile needs the sh_out of its neighbours toward the light, so a W x H block of tiles takes
// W + H - 1 waves). Arithmetic as the reference: fp32 with separate multiply/add (-fmad=false), the double-precision steps where the reference has them
// (get_xpos' "+ 0.5", dir_ratio, shadow_z).
#include "tw_internal.h"
#include <algorithm>
#include <map>
#include <vector>
#include <math.h>

namespace {

struct ShadowDev {
	float xs, ys, dx, dy, dxi, dyi, zmin, zmax; // X/Y_SCENE_SIZE, DX/DY_VAL, their inverses, clip z range
	float dirx, diry, dirz, dist;
	int dim; double dir_ratio;
};
struct Pt {float x, y, z;};

__device__ __forceinline__ int region_of(Pt v, const float (&d)[3][2]) { // get_region, src/inlines.h:522-528
	int r = 0;
	if (v.x < d[0][0]) {r |= 0x01;} else if (v.x >= d[0][1]) {r |= 0x02;}
	if (v.y < d[1][0]) {r |= 0x04;} else if (v.y >= d[1][1]) {r |= 0x08;}
	if (v.z < d[2][0]) {r |= 0x10;} else if (v.z >= d[2][1]) {r |= 0x20;}
	return r;
}
__device__ bool line_clip(Pt &v1, Pt &v2, const float (&d)[3][2]) { // do_line_clip, src/Math3d.cpp:1029-1034,1070-1086
	int const region1 = region_of(v1, d), region2 = region_of(v2, d);
	if (region1 & region2) return false;
	int const region3 = region1 | region2;
	if (region3 == 0) return true;
	float tmin = 0.0f, tmax = 1.0f;
	Pt const dv = {v2.x - v1.x, v2.y - v1.y, v2.z - v1.z};
#define TW_CLIP(reg, va, vb, vd, vc) if (region3 & (reg)) {float const t = __fdiv_rn((va) - (vb), (vd)); if ((vc) > 0.0f) {if (t > tmin) tmin = t;} else {if (t < tmax) tmax = t;} if (tmin >= tmax) return false;}
	TW_CLIP(0x01, d[0][0], v1.x, dv.x,  dv.x)
	TW_CLIP(0x02, d[0][1], v1.x, dv.x, -dv.x)
	TW_CLIP(0x04, d[1][0], v1.y, dv.y,  dv.y)
	TW_CLIP(0x08, d[1][1], v1.y, dv.y, -dv.y)
	TW_CLIP(0x10, d[2][0], v1.z, dv.z,  dv.z)
	TW_CLIP(0x20, d[2][1], v1.z, dv.z, -dv.z)
#undef TW_CLIP
	if (tmax > 1.0E-12f) {v2.x = v1.x + dv.x*tmax; v2.y = v1.y + dv.y*tmax; v2.z = v1.z + dv.z*tmax;}
	if ((double)tmin < (1.0 - (double)1.0E-12f)) {v1.x += dv.x*tmin; v1.y += dv.y*tmin; v1.z += dv.z*tmin;}
	return true;
}
__device__ __forceinline__ int to_pos(float v, float scene, float inv) {return (int)((double)((v + scene)*inv) + 0.5);} // get_xpos / get_ypos, src/mesh.h:129-130

__global__ void shadow_init_kernel(unsigned char *smask, unsigned long long *keys, size_t ncells, size_t nkeys, unsigned char val) {
	size_t const i = (size_t)blockIdx.x*blockDim.x + threadIdx.x, stride = (size_t)gridDim.x*blockDim.x;
	for (size_t k = i; k < ncells; k += stride) {smask[k] = val;}
	for (size_t k = i; k < nkeys; k += stride) {keys[k] = 0ull;}
}
// one thread per ray of one tile of the wave: blockIdx.y = position in the wave's tile list
__global__ void shadow_rays_kernel(const float *__restrict__ zvals, unsigned char *__restrict__ smask, int n, ShadowDev S, const int *__restrict__ wave_tiles,
	const int *__restrict__ nb_x, const int *__restrict__ nb_y, const float *__restrict__ ox, const float *__restrict__ oy, unsigned long long *__restrict__ kx, unsigned long long *__restrict__ ky)
{
	int const ray = blockIdx.x*blockDim.x + threadIdx.x;
	if (ray >= 4*n) return;
	int const tile = wave_tiles[blockIdx.y];
	const float *mh = zvals + (size_t)tile*n*n;
	const float *sh_in_x = (nb_y[tile] >= 0) ? ox + (size_t)nb_y[tile]*n : nullptr; // the y neighbour's sh_out[0] (src/tiled_mesh.cpp:680-686 with d = 1)
	const float *sh_in_y = (nb_x[tile] >= 0) ? oy + (size_t)nb_x[tile]*n : nullptr; // the x neighbour's sh_out[1] (d = 0)
	unsigned long long *out_x = kx + (size_t)tile*n, *out_y = ky + (size_t)tile*n;
	Pt v1;
	if (ray < 2*n) {v1.x = -S.xs + S.dx*(float)((S.dirx > 0.0f) ? 0 : n); v1.y = (float)((double)(-S.ys) + 0.5*(double)S.dy*(double)ray); v1.z = 0.0f;}       // run_x, :478-481
	else {int const x = ray - 2*n; v1.x = (float)((double)(-S.xs) + 0.5*(double)S.dx*(double)x); v1.y = -S.ys + S.dy*(float)((S.diry > 0.0f) ? 0 : n); v1.z = 0.0f;} // run_y, :482-485
	Pt v2 = {v1.x + S.dirx*S.dist, v1.y + S.diry*S.dist, v1.z + 0.0f};
	float const d[3][2] = {{-S.xs, -S.xs + S.dx*(float)n}, {-S.ys, -S.ys + S.dy*(float)n}, {S.zmin, S.zmax}};
	if (!line_clip(v1, v2, d)) return;
	int const xa = to_pos(v1.x, S.xs, S.dxi), ya = to_pos(v1.y, S.ys, S.dyi), xb = to_pos(v2.x, S.xs, S.dxi), yb = to_pos(v2.y, S.ys, S.dyi), ddx = xb - xa, ddy = yb - ya;
	bool inited = false;
	Pt cur = {0.0f, 0.0f, 0.0f};
	int x = xa, y = ya, dx1 = 0, dy1 = 0, dx2 = 0, dy2 = 0; // Bresenham, :429-440
	if (ddx < 0) {dx1 = -1; dx2 = -1;} else if (ddx > 0) {dx1 = 1; dx2 = 1;}
	if (ddy < 0) {dy1 = -1;} else if (ddy > 0) {dy1 = 1;}
	int longest = abs(ddx), shortest = abs(ddy);
	if (longest <= shortest) {
		int const t = longest; longest = shortest; shortest = t;
		if (ddy < 0) {dy2 = -1;} else if (ddy > 0) {dy2 = 1;}
		dx2 = 0;
	}
	int numerator = longest >> 1;
	unsigned long long const seq = (unsigned long long)(ray + 1) << 32;
	for (int i = 0; i <= longest; i++) {
		if (x >= 0 && y >= 0 && x < n && y < n) {
			Pt const pt = {-S.xs + S.dx*(float)x, -S.ys + S.dy*(float)y, __ldg(mh + y*n + x)};
			if (sh_in_y != nullptr && x == xa && sh_in_y[y] > TW_MESH_MIN_Z) {cur.x = pt.x; cur.y = pt.y; cur.z = sh_in_y[y]; inited = true;}      // starting shadow height
			else if (sh_in_x != nullptr && y == ya && sh_in_x[x] > TW_MESH_MIN_Z) {cur.x = pt.x; cur.y = pt.y; cur.z = sh_in_x[x]; inited = true;}
			float const shadow_z = (float)((double)((S.dim ? pt.y : pt.x) - (S.dim ? cur.y : cur.x))*S.dir_ratio + (double)cur.z);
			if (inited && shadow_z > pt.z) { // shadowed
				size_t const c = (size_t)tile*n*n + (size_t)y*n + x; // byte index in the whole (4-byte aligned) mask: a tile of odd size starts mid-word
				atomicOr((unsigned *)(smask + (c & ~(size_t)3)), (unsigned)TW_MESH_SHADOW << ((unsigned)(c & 3)*8u));
				if (x == xb) {atomicMax(out_y + y, seq | __float_as_uint(shadow_z));}
				if (y == yb) {atomicMax(out_x + x, seq | __float_as_uint(shadow_z));}
			}
			else {cur = pt;}
			inited = true;
		}
		numerator += shortest;
		if (numerator >= longest) {numerator -= longest; x += dx1; y += dy1;} else {x += dx2; y += dy2;}
	}
}
__global__ void shadow_unpack_kernel(const unsigned long long *__restrict__ kx, const unsigned long long *__restrict__ ky, float *__restrict__ ox, float *__restrict__ oy, int n, const int *__restrict__ wave_tiles) {
	int const i = blockIdx.x*blockDim.x + threadIdx.x;
	if (i >= n) return;
	size_t const o = (size_t)wave_tiles[blockIdx.y]*n + i;
	unsigned long long const a = kx[o], b = ky[o];
	ox[o] = a ? __uint_as_float((unsigned)a) : TW_MESH_MIN_Z; // sh_out starts at MESH_MIN_Z (src/tiled_mesh.cpp:677)
	oy[o] = b ? __uint_as_float((unsigned)b) : TW_MESH_MIN_Z;
}

} // namespace

extern "C" int tw_tile_shadows_batch(tw_ctx *ctx, const float *zvals, const int32_t *tile_xy, uint32_t ntiles, uint32_t zvsize, const tw_shadow_params *sp,
                                     uint8_t *smask, float *sh_out_x, float *sh_out_y)
{
	int rc = tw_enter(ctx); if (rc) return rc;
	if (!zvals || !tile_xy || !sp || !smask || ntiles == 0 || zvsize < 2) return tw_set_error(ctx, TW_ERR_ARG, "null argument, no tiles or zvsize < 2");
	if (ntiles > 65535) return tw_set_error(ctx, TW_ERR_ARG, "at most 65535 tiles per call");
	int const n = (int)zvsize;
	size_t const cells = (size_t)ntiles*n*n, edge = (size_t)ntiles*n;
	// neighbours toward the light, dependency waves
	int const sx = (sp->lpos[0] < 0.0f) ? -1 : 1, sy = (sp->lpos[1] < 0.0f) ? -1 : 1;
	std::map<std::pair<int, int>, int> where;
	for (uint32_t t = 0; t < ntiles; ++t) {where[std::make_pair(tile_xy[2*t], tile_xy[2*t+1])] = (int)t;}
	std::vector<int> nbx(ntiles, -1), nby(ntiles, -1), level(ntiles, -1);
	for (uint32_t t = 0; t < ntiles; ++t) {
		auto a = where.find(std::make_pair(tile_xy[2*t] + sx, tile_xy[2*t+1])); if (a != where.end()) nbx[t] = a->second;
		auto b = where.find(std::make_pair(tile_xy[2*t], tile_xy[2*t+1] + sy)); if (b != where.end()) nby[t] = b->second;
	}
	int nlevels = 0;
	{ // level = longest chain of neighbours toward the light (they form a DAG: every edge moves one step toward the light)
		std::vector<int> order(ntiles);
		for (uint32_t t = 0; t < ntiles; ++t) order[t] = (int)t;
		std::sort(order.begin(), order.end(), [&](int a, int b) {return (sx*tile_xy[2*a] + sy*tile_xy[2*a+1]) > (sx*tile_xy[2*b] + sy*tile_xy[2*b+1]);}); // closest to the light first
		for (int t : order) {
			int l = 0;
			if (nbx[t] >= 0) l = std::max(l, level[nbx[t]] + 1);
			if (nby[t] >= 0) l = std::max(l, level[nby[t]] + 1);
			level[t] = l; nlevels = std::max(nlevels, l + 1);
		}
	}
	std::vector<int> wave_tiles; std::vector<int> wave_start(nlevels + 1, 0);
	for (int l = 0; l < nlevels; ++l) {for (uint32_t t = 0; t < ntiles; ++t) {if (level[t] == l) wave_tiles.push_back((int)t);} wave_start[l + 1] = (int)wave_tiles.size();}
	// light direction and ray length (mesh_shadow_gen::run, :492-496), on the host with the reference's operations
	ShadowDev S;
	memset(&S, 0, sizeof(S));
	S.xs = sp->x_scene_size; S.ys = sp->y_scene_size; S.dx = sp->dx_val; S.dy = sp->dy_val; S.dxi = sp->dx_val_inv; S.dyi = sp->dy_val_inv; S.zmin = sp->zmin; S.zmax = sp->zmax;
	bool const all_shadowed = (!sp->no_shadow && sp->lpos[2] < sp->zmin);
	bool const trace = !(sp->no_shadow || (sp->lpos[0] == 0.0f && sp->lpos[1] == 0.0f));
	if (trace) {
		volatile float m2 = sp->lpos[0]*sp->lpos[0]; volatile float m2b = sp->lpos[1]*sp->lpos[1]; volatile float m2c = sp->lpos[2]*sp->lpos[2];
		volatile float ms = m2 + m2b; ms = ms + m2c;
		float const vmag = sqrtf(ms);
		float nx = sp->lpos[0], ny = sp->lpos[1], nz = sp->lpos[2];
		if (!(vmag < 1.0E-12f)) {nx = sp->lpos[0]/vmag; ny = sp->lpos[1]/vmag; nz = sp->lpos[2]/vmag;} // get_norm
		S.dirx = -nx; S.diry = -ny; S.dirz = -nz;
		volatile float q1 = S.dirx*S.dirx; volatile float q2 = S.diry*S.diry; volatile float q = q1 + q2;
		S.dist = (float)(2.0*sp->xy_sum_size/sqrtf(q));
		S.dim = (fabsf(S.dirx) < fabsf(S.diry)) ? 1 : 0;
		S.dir_ratio = (double)(S.dirz/(S.dim ? S.diry : S.dirx));
	}
	size_t const nkeys = tw_align256(edge*sizeof(unsigned long long))/sizeof(unsigned long long); // keys of sh_out_x, then those of sh_out_y
	const float *d_z; uint8_t *d_m; unsigned long long *d_kx; float *d_ox, *d_oy; const int *d_wave, *d_nbx, *d_nby;
	tw_stage st(ctx);
	st.in(&d_z, zvals, cells*sizeof(float));
	st.out(&d_m, smask, cells, 4); // + 4: the rays set flag bytes with atomics on the 32-bit word that holds them
	st.temp(&d_kx, 2*nkeys*sizeof(unsigned long long));
	st.temp(&d_ox, edge*sizeof(float));
	st.temp(&d_oy, edge*sizeof(float));
	st.in(&d_wave, wave_tiles.data(), (size_t)ntiles*sizeof(int));
	st.in(&d_nbx, nbx.data(), (size_t)ntiles*sizeof(int));
	st.in(&d_nby, nby.data(), (size_t)ntiles*sizeof(int));
	rc = st.commit(); if (rc) return rc;
	if ((size_t)d_m & 3) return tw_set_error(ctx, TW_ERR_ARG, "smask must be 4-byte aligned (flag bytes are set with 32-bit atomics)"); // only a device buffer can be
	unsigned long long *d_ky = d_kx + nkeys;
	shadow_init_kernel<<<148*8, 256, 0, ctx->stream>>>(d_m, d_kx, cells, 2*nkeys, all_shadowed ? (unsigned char)TW_MESH_SHADOW : (unsigned char)0);
	TW_LAUNCH_CHECK(ctx);
	for (int l = 0; l < nlevels; ++l) {
		int const nw = wave_start[l + 1] - wave_start[l];
		if (trace) {
			shadow_rays_kernel<<<dim3((4*n + 127)/128, nw), 128, 0, ctx->stream>>>(d_z, d_m, n, S, d_wave + wave_start[l], d_nbx, d_nby, d_ox, d_oy, d_kx, d_ky);
			TW_LAUNCH_CHECK(ctx);
		}
		shadow_unpack_kernel<<<dim3((n + 127)/128, nw), 128, 0, ctx->stream>>>(d_kx, d_ky, d_ox, d_oy, n, d_wave + wave_start[l]);
		TW_LAUNCH_CHECK(ctx);
	}
	if (sh_out_x) {TW_CUDA(ctx, cudaMemcpyAsync(sh_out_x, d_ox, edge*sizeof(float), cudaMemcpyDefault, ctx->stream));}
	if (sh_out_y) {TW_CUDA(ctx, cudaMemcpyAsync(sh_out_y, d_oy, edge*sizeof(float), cudaMemcpyDefault, ctx->stream));}
	return st.finish();
}
