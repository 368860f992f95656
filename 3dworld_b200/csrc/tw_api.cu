// tw_api.cu - the extern "C" boundary (include/tw3d.h): context management, host/device pointer staging, and dispatch to the kernels.
// There is deliberately NO CPU path in this library: without a CUDA device tw_create fails and nothing else can be called.
#include "tw_internal.h"
#include <algorithm>
#include <stdarg.h>
#include <stdlib.h>
#include <new>
#include <vector>
#include <math.h>

extern "C" void twi_build_dir_table(float *cs2x1e6);

int tw_set_error(tw_ctx *ctx, int status, const char *fmt, ...) {
	if (ctx) {
		va_list ap; va_start(ap, fmt);
		vsnprintf(ctx->err, sizeof(ctx->err), fmt, ap);
		va_end(ap);
	}
	return status;
}

int tw_reserve(tw_ctx *ctx, int slot, size_t bytes) {
	if (ctx->scratch_bytes[slot] >= bytes) return TW_OK;
	TW_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	if (ctx->d_scratch[slot]) {TW_CUDA(ctx, cudaFree(ctx->d_scratch[slot])); ctx->d_scratch[slot] = nullptr; ctx->scratch_bytes[slot] = 0;}
	size_t const rounded = (bytes + ((size_t)1 << 20) - 1) & ~(((size_t)1 << 20) - 1);
	TW_CUDA(ctx, cudaMalloc(&ctx->d_scratch[slot], rounded));
	ctx->scratch_bytes[slot] = rounded;
	return TW_OK;
}

int tw_reserve_pinned(tw_ctx *ctx, size_t bytes) {
	if (ctx->pinned_bytes >= bytes) return TW_OK;
	TW_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	if (ctx->h_pinned) {TW_CUDA(ctx, cudaFreeHost(ctx->h_pinned)); ctx->h_pinned = nullptr; ctx->pinned_bytes = 0;}
	TW_CUDA(ctx, cudaMallocHost(&ctx->h_pinned, bytes));
	ctx->pinned_bytes = bytes;
	return TW_OK;
}

bool tw_is_device_ptr(const void *p) {
	cudaPointerAttributes a;
	if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {cudaGetLastError(); return false;}
	return (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged);
}

bool tw_stage::add(void *d, const void *caller, size_t bytes, size_t slack, int dir) {
	bool const host = (dir & TEMP) || is_host(caller);
	if (n_ < MAX_BUFFERS) {e_[n_] = entry{d, caller, nullptr, bytes, host ? tw_align256(bytes + slack) : 0, host ? dir : 0, host};}
	++n_; // commit() rejects more than MAX_BUFFERS
	return host;
}

int tw_stage::commit() {
	if (n_ > MAX_BUFFERS) return tw_set_error(ctx_, TW_ERR_STATE, "tw_stage: more than %d buffers", (int)MAX_BUFFERS);
	size_t total = 0;
	for (int i = 0; i < n_; ++i) {total += e_[i].region;}
	if (total) {
		if (ctx_->scratch0_held) return tw_set_error(ctx_, TW_ERR_STATE, "scratch slot 0 holds the buffers of the calling entry point: a nested call must pass device pointers");
		int const rc = tw_reserve(ctx_, 0, total); if (rc) return rc;
		held_ = ctx_->scratch0_held = true;
	}
	char *q = (char *)ctx_->d_scratch[0];
	for (int i = 0; i < n_; ++i) {
		entry &e = e_[i];
		e.dev = e.host ? (void *)q : const_cast<void *>(e.caller);
		memcpy(e.d, &e.dev, sizeof(void *)); // e.d is the call site's T* variable
		q += e.region;
		if (e.dir & IN) {TW_CUDA(ctx_, cudaMemcpyAsync(e.dev, e.caller, e.bytes, cudaMemcpyHostToDevice, ctx_->stream));}
	}
	return TW_OK;
}

int tw_stage::finish() {
	for (int i = 0; i < n_; ++i) {
		entry const &e = e_[i];
		if (e.dir & OUT) {TW_CUDA(ctx_, cudaMemcpyAsync(const_cast<void *>(e.caller), e.dev, e.bytes, cudaMemcpyDeviceToHost, ctx_->stream));}
	}
	TW_CUDA(ctx_, cudaStreamSynchronize(ctx_->stream));
	return TW_OK;
}

int twi_ensure_aux_streams(tw_ctx *ctx) {
	if (ctx->aux_stream[0]) return TW_OK;
	int lo = 0, hi = 0; // the latency-bound droplet kernels / band copies get the higher priority
	TW_CUDA(ctx, cudaDeviceGetStreamPriorityRange(&lo, &hi));
	bool const prio = !(getenv("TW_PIPE_NOPRIO"));
	for (int i = 0; i < 3; ++i) {TW_CUDA(ctx, cudaStreamCreateWithPriority(&ctx->aux_stream[i], cudaStreamNonBlocking, prio ? hi : lo));}
	return TW_OK;
}

namespace {

// slot-2 layout (small device scalars)
constexpr size_t OFF_MM = 0, OFF_BAD = 64, OFF_TILES = 4096;

int check_ctx(tw_ctx *ctx) { // NOTE: makes ctx->device the calling thread's current CUDA device and leaves it so (documented in tw3d.h: one context per thread)
	if (!ctx) return TW_ERR_ARG;
	cudaError_t e = cudaSetDevice(ctx->device);
	if (e != cudaSuccess) return tw_set_error(ctx, TW_ERR_CUDA, "cudaSetDevice(%d): %s", ctx->device, cudaGetErrorString(e));
	return TW_OK;
}

int single_minmax(tw_ctx *ctx, unsigned **d_mm) { // the one (min, max) pair of slot 2, initialised for a reduction
	int const rc = tw_reserve(ctx, 2, OFF_TILES); if (rc) return rc;
	*d_mm = (unsigned *)((char *)ctx->d_scratch[2] + OFF_MM);
	return twi_init_minmax(ctx, *d_mm, 1);
}

// setup_height_gen_async / build_arrays((x1 - MESH_X_SIZE/2), (y1 - MESH_Y_SIZE/2), dx, dy, ...): int -> float, then mx0 = dx*x0 (src/tiled_mesh.cpp:461, src/mesh_gen.cpp:591)
std::vector<float2> tile_origins(const int32_t *origins_xy, uint32_t ntiles, int mesh_x_size, int mesh_y_size, float dx, float dy) {
	std::vector<float2> org(ntiles);
	for (uint32_t t = 0; t < ntiles; ++t) {
		float const x0 = (float)(origins_xy[2*t] - mesh_x_size/2), y0 = (float)(origins_xy[2*t+1] - mesh_y_size/2);
		org[t] = make_float2(dx*x0, dy*y0);
	}
	return org;
}

int read_minmax(tw_ctx *ctx, const unsigned *d_mm, tw_minmax *mm, uint32_t n) { // synchronous
	int rc = tw_reserve_pinned(ctx, (size_t)n*2*sizeof(unsigned));
	if (rc) return rc;
	TW_CUDA(ctx, cudaMemcpyAsync(ctx->h_pinned, d_mm, (size_t)n*2*sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream));
	TW_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	unsigned const *u = (unsigned const *)ctx->h_pinned;
	for (uint32_t i = 0; i < n; ++i) {mm[i].zmin = tw_ord2f(u[2*i]); mm[i].zmax = tw_ord2f(u[2*i+1]);}
	return TW_OK;
}

int validate_height(tw_ctx *ctx, const tw_grid2d *g, const tw_height_params *p, const float *out) {
	if (!g || !p || !out) return tw_set_error(ctx, TW_ERR_ARG, "null argument");
	if (g->nx == 0 || g->ny == 0) return tw_set_error(ctx, TW_ERR_ARG, "nx, ny must be > 0 (reference asserts, src/mesh_gen.cpp:589)");
	if (p->gen_mode < 0 || p->gen_mode > TW_MGEN_DWARP_GPU) return tw_set_error(ctx, TW_ERR_ARG, "bad gen_mode %d", p->gen_mode);
	if (p->start_eval_sin < 0 || p->start_eval_sin > TW_F_TABLE_SIZE) return tw_set_error(ctx, TW_ERR_ARG, "start_eval_sin out of range (src/mesh_gen.cpp:590)");
	if (!ctx->have_sin) return tw_set_error(ctx, TW_ERR_STATE, "tw_set_sin_table() has not been called");
	return TW_OK;
}

} // namespace

int tw_enter(tw_ctx *ctx) {
	int const rc = check_ctx(ctx); if (rc) return rc;
	if (ctx->async.pending) {return tw_heightgen_2d_poll(ctx, 1);} // an outstanding tw_heightgen_2d_launch completes before other work reuses the scratch buffers
	return TW_OK;
}

extern "C" {

int tw_abi_version(void) {return TW_ABI_VERSION;}

int tw_create(int device, tw_ctx **out) {
	if (!out) return TW_ERR_ARG;
	*out = nullptr;
	int ndev = 0;
	if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {cudaGetLastError(); return TW_ERR_NO_DEVICE;}
	if (device < 0 || device >= ndev) return TW_ERR_ARG;
	if (cudaSetDevice(device) != cudaSuccess) {cudaGetLastError(); return TW_ERR_CUDA;}
	tw_ctx *ctx = new (std::nothrow) tw_ctx();
	if (!ctx) return TW_ERR_CUDA;
	ctx->device = device;
	if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {delete ctx; cudaGetLastError(); return TW_ERR_CUDA;}
	if (cudaEventCreateWithFlags(&ctx->async.done, cudaEventDisableTiming) != cudaSuccess) {cudaStreamDestroy(ctx->stream); delete ctx; cudaGetLastError(); return TW_ERR_CUDA;}
	*out = ctx;
	return TW_OK;
}

void tw_destroy(tw_ctx *ctx) {
	if (!ctx) return;
	if (ctx->dist) tw_dist_finalize(ctx);
	cudaSetDevice(ctx->device);
	cudaStreamSynchronize(ctx->stream);
	for (int i = 0; i < 3; ++i) {if (ctx->d_scratch[i]) cudaFree(ctx->d_scratch[i]);}
	if (ctx->d_sin_table) cudaFree(ctx->d_sin_table);
	if (ctx->d_dir_table) cudaFree(ctx->d_dir_table);
	if (ctx->d_simplex_lut) cudaFree(ctx->d_simplex_lut);
	if (ctx->d_glm3_lut) cudaFree(ctx->d_glm3_lut);
	if (ctx->d_sine_params) cudaFree(ctx->d_sine_params);
	if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
	if (ctx->async.done) cudaEventDestroy(ctx->async.done);
	for (int i = 0; i < 3; ++i) {if (ctx->aux_stream[i]) cudaStreamDestroy(ctx->aux_stream[i]);}
	for (int i = 0; i < 4; ++i) {
		if (ctx->heavy_stream[i]) cudaStreamDestroy(ctx->heavy_stream[i]);
		if (ctx->ev_fork[i]) cudaEventDestroy(ctx->ev_fork[i]);
		if (ctx->ev_join[i]) cudaEventDestroy(ctx->ev_join[i]);
	}
	cudaStreamDestroy(ctx->stream);
	delete ctx;
}

const char *tw_last_error(const tw_ctx *ctx) {return ctx ? ctx->err : "null context";}
void *tw_stream(tw_ctx *ctx) {return ctx ? (void *)ctx->stream : nullptr;}
uint64_t tw_launch_count(const tw_ctx *ctx) {return ctx ? ctx->launches : 0;}
uint64_t tw_last_erosion_steps(const tw_ctx *ctx) {return ctx ? ctx->last_erosion_steps : 0;}

int tw_sync(tw_ctx *ctx) {
	int rc = check_ctx(ctx); if (rc) return rc;
	TW_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	return TW_OK;
}

int tw_set_sin_table(tw_ctx *ctx, const float *tab) {
	int rc = check_ctx(ctx); if (rc) return rc;
	std::vector<float> built;
	if (!tab) {built.resize(TW_SIN_TABLE_SIZE); tw_build_sin_table(built.data()); tab = built.data();}
	if (!ctx->d_sin_table) {TW_CUDA(ctx, cudaMalloc(&ctx->d_sin_table, TW_SIN_TABLE_SIZE*sizeof(float)));}
	TW_CUDA(ctx, cudaMemcpyAsync(ctx->d_sin_table, tab, TW_SIN_TABLE_SIZE*sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
	if (!ctx->d_dir_table) {
		std::vector<float> dir(2*1000000);
		twi_build_dir_table(dir.data());
		TW_CUDA(ctx, cudaMalloc(&ctx->d_dir_table, dir.size()*sizeof(float)));
		TW_CUDA(ctx, cudaMemcpyAsync(ctx->d_dir_table, dir.data(), dir.size()*sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
		TW_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	}
	TW_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	ctx->have_sin = true;
	return TW_OK;
}

int tw_set_sine_params(tw_ctx *ctx, const float *sp) {
	int rc = check_ctx(ctx); if (rc) return rc;
	if (!sp) return tw_set_error(ctx, TW_ERR_ARG, "null sine_params");
	if (!ctx->d_sine_params) {TW_CUDA(ctx, cudaMalloc(&ctx->d_sine_params, TW_F_TABLE_SIZE*5*sizeof(float)));}
	memcpy(ctx->h_sine_params, sp, sizeof(ctx->h_sine_params));
	TW_CUDA(ctx, cudaMemcpyAsync(ctx->d_sine_params, ctx->h_sine_params, sizeof(ctx->h_sine_params), cudaMemcpyHostToDevice, ctx->stream));
	TW_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	ctx->have_sine_params = true;
	return TW_OK;
}

// ------------------------------------------------------------------------------------------------ 2-D height
int tw_heightgen_2d_launch(tw_ctx *ctx, const tw_grid2d *g, const tw_height_params *p, int enable_glaciate, int min_start_sin, float *out, tw_minmax *mm) {
	int rc = tw_enter(ctx); if (rc) return rc;
	rc = validate_height(ctx, g, p, out); if (rc) return rc;
	float *d_out;
	tw_stage st(ctx);
	bool const host_out = st.view(&d_out, out, (size_t)g->nx*g->ny*sizeof(float));
	rc = st.commit(); if (rc) return rc;
	unsigned *d_mm = nullptr;
	if (mm) {rc = single_minmax(ctx, &d_mm); if (rc) return rc;}
	if (host_out) {rc = twi_ensure_aux_streams(ctx); if (rc) return rc;}
	rc = twi_heightgen(ctx, g, p, enable_glaciate, min_start_sin, nullptr, 1, d_out, d_mm, host_out ? out : nullptr); // host out: band-wise D2H overlapped with compute
	if (rc) return rc;
	if (mm) {
		rc = tw_reserve_pinned(ctx, 2*sizeof(unsigned)); if (rc) return rc;
		TW_CUDA(ctx, cudaMemcpyAsync(ctx->h_pinned, d_mm, 2*sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream));
	}
	TW_CUDA(ctx, cudaEventRecord(ctx->async.done, ctx->stream));
	ctx->async.pending = true; ctx->async.host_mm = mm; ctx->async.n_mm = mm ? 1 : 0;
	return TW_OK;
}

int tw_heightgen_2d_poll(tw_ctx *ctx, int wait) {
	int rc = check_ctx(ctx); if (rc) return rc;
	if (!ctx->async.pending) return TW_OK;
	if (wait) {TW_CUDA(ctx, cudaEventSynchronize(ctx->async.done));}
	else {
		cudaError_t const e = cudaEventQuery(ctx->async.done);
		if (e == cudaErrorNotReady) return TW_ERR_NOT_READY;
		if (e != cudaSuccess) return tw_set_error(ctx, TW_ERR_CUDA, "cudaEventQuery: %s", cudaGetErrorString(e));
	}
	ctx->async.pending = false;
	if (ctx->async.host_mm) {
		unsigned const *u = (unsigned const *)ctx->h_pinned;
		ctx->async.host_mm->zmin = tw_ord2f(u[0]); ctx->async.host_mm->zmax = tw_ord2f(u[1]);
		ctx->async.host_mm = nullptr;
	}
	cudaError_t const e = cudaGetLastError();
	if (e != cudaSuccess) return tw_set_error(ctx, TW_ERR_CUDA, "async height generation failed: %s", cudaGetErrorString(e));
	return TW_OK;
}

int tw_heightgen_2d(tw_ctx *ctx, const tw_grid2d *g, const tw_height_params *p, int enable_glaciate, int min_start_sin, float *out, tw_minmax *mm) {
	int rc = tw_heightgen_2d_launch(ctx, g, p, enable_glaciate, min_start_sin, out, mm);
	if (rc) return rc;
	return tw_heightgen_2d_poll(ctx, 1);
}

// tile_t::create_texture, terrain part (include/tw3d.h): the jitter noise grid of every tile (force-sine-mode build_arrays at 80x the cell size, start index >= 50,
// no glaciate) with the batched sine-tile generator, then one thread per texel
int tw_tile_weights_batch(tw_ctx *ctx, const float *zvals, const int32_t *origins_xy, uint32_t ntiles, int mesh_x_size, int mesh_y_size, float dx, float dy,
                          uint32_t zvsize, const tw_height_params *p, const tw_weight_params *wp, const float *tile_params, uint8_t *weights, uint8_t *has_any_grass)
{
	int rc = tw_enter(ctx); if (rc) return rc;
	if (!zvals || !origins_xy || !p || !wp || !tile_params || !weights || ntiles == 0 || zvsize < 3) return tw_set_error(ctx, TW_ERR_ARG, "tw_tile_weights_batch: null argument, no tiles or zvsize < 3");
	tw_weight_params W = *wp;
	int seen[5] = {0, 0, 0, 0, 0};
	for (int i = 0; i < 5; ++i) {
		if (W.tex_class[i] < 0 || W.tex_class[i] > 4 || seen[W.tex_class[i]]++) return tw_set_error(ctx, TW_ERR_ARG, "tex_class must name each ground texture exactly once (get_texture_ixs asserts it)");
		W.class_ix[W.tex_class[i]] = i;
	}
	if (!(W.zmax > W.zmin)) return tw_set_error(ctx, TW_ERR_ARG, "zmax must exceed zmin");
	uint32_t const stride = zvsize - 1;
	size_t const zn = (size_t)ntiles*zvsize*zvsize, tn = (size_t)ntiles*stride*stride;
	float *d_rand; const float *d_z, *d_p; uint8_t *d_w, *d_f;
	tw_stage st(ctx);
	st.temp(&d_rand, tn*sizeof(float));
	st.in(&d_z, zvals, zn*sizeof(float));
	st.out(&d_w, weights, tn*4);
	st.out(&d_f, has_any_grass, ntiles);
	st.in(&d_p, tile_params, (size_t)ntiles*8*sizeof(float));
	rc = st.commit(); if (rc) return rc;
	if (d_f) {TW_CUDA(ctx, cudaMemsetAsync(d_f, 0, ntiles, ctx->stream));}
	// height_gen.build_arrays((x1 - MESH_X_SIZE/2), (y1 - MESH_Y_SIZE/2), MESH_NOISE_FREQ*DX_VAL, MESH_NOISE_FREQ*DY_VAL, tsize, tsize, 0, 1) (src/tiled_mesh.cpp:1103)
	float const MESH_NOISE_FREQ = 80.0f;
	tw_grid2d g; g.x0 = 0; g.y0 = 0; g.dx = MESH_NOISE_FREQ*dx; g.dy = MESH_NOISE_FREQ*dy; g.nx = stride; g.ny = stride;
	std::vector<float2> const org = tile_origins(origins_xy, ntiles, mesh_x_size, mesh_y_size, g.dx, g.dy);
	tw_height_params ps = *p;
	ps.gen_mode = TW_MGEN_SINE; ps.gen_shape = 0; // force_sine_mode: gen_mode = MGEN_SINE, gen_shape = 0 (src/mesh_gen.cpp:592-593)
	rc = twi_heightgen_sine_tiles(ctx, &g, &ps, 0, 50, org.data(), ntiles, d_rand, nullptr);
	if (rc) return rc;
	rc = twi_tile_weights(ctx, d_z, d_rand, ntiles, zvsize, d_p, &W, d_w, d_f);
	if (rc) return rc;
	return st.finish();
}

int tw_heightgen_tiles(tw_ctx *ctx, const int32_t *origins_xy, uint32_t ntiles, int mesh_x_size, int mesh_y_size, float dx, float dy,
                       uint32_t zvsize, const tw_height_params *p, float *out, tw_minmax *mm)
{
	int rc = tw_enter(ctx); if (rc) return rc;
	if (!origins_xy || ntiles == 0) return tw_set_error(ctx, TW_ERR_ARG, "no tiles");
	tw_grid2d g; g.x0 = 0; g.y0 = 0; g.dx = dx; g.dy = dy; g.nx = zvsize; g.ny = zvsize;
	rc = validate_height(ctx, &g, p, out); if (rc) return rc;
	size_t const tile_elems = (size_t)zvsize*zvsize;
	float *d_out;
	tw_stage st(ctx);
	st.out(&d_out, out, tile_elems*ntiles*sizeof(float));
	rc = st.commit(); if (rc) return rc;
	size_t const mm_bytes = (size_t)ntiles*2*sizeof(unsigned), org_bytes = (size_t)ntiles*sizeof(float2);
	rc = tw_reserve(ctx, 2, OFF_TILES + mm_bytes + org_bytes); if (rc) return rc;
	unsigned *d_mm = mm ? (unsigned *)((char *)ctx->d_scratch[2] + OFF_TILES) : nullptr;
	float2 *d_org = (float2 *)((char *)ctx->d_scratch[2] + OFF_TILES + mm_bytes);
	if (d_mm) {rc = twi_init_minmax(ctx, d_mm, ntiles); if (rc) return rc;}
	std::vector<float2> const org = tile_origins(origins_xy, ntiles, mesh_x_size, mesh_y_size, dx, dy);
	if (p->gen_mode != TW_MGEN_SINE) {
		TW_CUDA(ctx, cudaMemcpyAsync(d_org, org.data(), org_bytes, cudaMemcpyHostToDevice, ctx->stream));
		TW_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); // org is a local vector
		uint32_t const zmax = 65535;
		for (uint32_t t0 = 0; t0 < ntiles; t0 += zmax) { // gridDim.z limit
			uint32_t const nt = (ntiles - t0 < zmax) ? ntiles - t0 : zmax;
			rc = twi_heightgen(ctx, &g, p, 1, 0, d_org + t0, nt, d_out + (size_t)t0*tile_elems, d_mm ? d_mm + 2*(size_t)t0 : nullptr);
			if (rc) return rc;
		}
	}
	else { // sine tables depend on the tile origin only through its column / row: W + H tables for a W x H block of tiles, one grid launch for the batch
		rc = twi_heightgen_sine_tiles(ctx, &g, p, 1, 0, org.data(), ntiles, d_out, d_mm);
		if (rc) return rc;
	}
	if (mm) {rc = read_minmax(ctx, d_mm, mm, ntiles); if (rc) return rc;}
	return st.finish();
}

// ------------------------------------------------------------------------------------------------ callers' tails
int tw_tile_bounds_batch(tw_ctx *ctx, const float *zvals, uint32_t ntiles, uint32_t zvsize, float wpz_max, float dx_val, float dy_val, uint32_t size, tw_tile_bounds *out) {
	int rc = tw_enter(ctx); if (rc) return rc;
	if (!zvals || !out || ntiles == 0 || zvsize < 4) return tw_set_error(ctx, TW_ERR_ARG, "null/empty argument");
	if (4*(zvsize/4) >= zvsize) return tw_set_error(ctx, TW_ERR_ARG, "zvsize %u: the last sub-block would end at cell %u (the reference asserts x_end < zvsize, src/tiled_mesh.cpp:520)", zvsize, 4*(zvsize/4));
	if (ntiles > 65535) return tw_set_error(ctx, TW_ERR_ARG, "at most 65535 tiles per call");
	struct Sub {float zmin, zmax; int wx1, wy1, wx2, wy2;};
	std::vector<Sub> sub((size_t)ntiles*16);
	const float *d_z; Sub *d_sub;
	tw_stage st(ctx);
	st.in(&d_z, zvals, (size_t)ntiles*zvsize*zvsize*sizeof(float));
	st.temp(&d_sub, sub.size()*sizeof(Sub));
	rc = st.commit(); if (rc) return rc;
	rc = twi_tile_bounds(ctx, d_z, ntiles, zvsize, wpz_max, d_sub); if (rc) return rc;
	TW_CUDA(ctx, cudaMemcpyAsync(sub.data(), d_sub, sub.size()*sizeof(Sub), cudaMemcpyDeviceToHost, ctx->stream));
	rc = st.finish(); if (rc) return rc;
	for (uint32_t t = 0; t < ntiles; ++t) { // combine the 16 sub-blocks exactly as the reference's loop does (src/tiled_mesh.cpp:517-540)
		tw_tile_bounds &b = out[t];
		b.mzmin = 100.0f; b.mzmax = -100.0f; b.mesh_dz = 0.0f; // FAR_DISTANCE
		b.wx1 = b.wy1 = 2147483647; b.wx2 = b.wy2 = -1;
		for (int k = 0; k < 16; ++k) {
			Sub const &q = sub[(size_t)t*16 + k];
			b.sub_zmin[k] = q.zmin; b.sub_zmax[k] = q.zmax;
			float const range = q.zmax - q.zmin;
			b.mesh_dz = (b.mesh_dz < range) ? range : b.mesh_dz;      // max_eq(mesh_dz, (szmax - szmin))
			b.mzmin = (q.zmin < b.mzmin) ? q.zmin : b.mzmin;          // min(mzmin, szmin)
			b.mzmax = (b.mzmax < q.zmax) ? q.zmax : b.mzmax;          // max(mzmax, szmax)
			if (q.wx1 < b.wx1) b.wx1 = q.wx1; if (q.wy1 < b.wy1) b.wy1 = q.wy1;
			if (q.wx2 > b.wx2) b.wx2 = q.wx2; if (q.wy2 > b.wy2) b.wy2 = q.wy2;
		}
		float const dz = b.mzmax - b.mzmin;
		b.radius = 0.5*sqrtf((dx_val*dx_val + dy_val*dy_val)*size*size + dz*dz); // src/tiled_mesh.cpp:541
	}
	return TW_OK;
}

int tw_glaciate_mesh(tw_ctx *ctx, float *mesh, int nx, int ny, int xoff2, int yoff2, int mesh_x_size, int mesh_y_size, const tw_height_params *p, tw_minmax *zbottom_ztop) {
	int rc = tw_enter(ctx); if (rc) return rc;
	if (!mesh || !p || nx <= 0 || ny <= 0 || ny > 65535) return tw_set_error(ctx, TW_ERR_ARG, "bad argument");
	if (!ctx->have_sin) return tw_set_error(ctx, TW_ERR_STATE, "tw_set_sin_table() has not been called");
	float *d_mesh;
	tw_stage st(ctx);
	st.inout(&d_mesh, mesh, (size_t)nx*ny*sizeof(float));
	rc = st.commit(); if (rc) return rc;
	unsigned *d_mm;
	rc = single_minmax(ctx, &d_mm); if (rc) return rc;
	rc = twi_glaciate_mesh(ctx, d_mesh, nx, ny, xoff2, yoff2, mesh_x_size, mesh_y_size, p, d_mm); if (rc) return rc;
	if (zbottom_ztop) {rc = read_minmax(ctx, d_mm, zbottom_ztop, 1); if (rc) return rc;}
	return st.finish();
}

// ------------------------------------------------------------------------------------------------ erosion
int tw_erode_tiles(tw_ctx *ctx, float *maps, uint32_t ntiles, int xsize, int ysize, const float *min_zvals, float min_zval_all,
                   uint32_t num_iters, const tw_erosion_params *p)
{
	int rc = tw_enter(ctx); if (rc) return rc;
	if (!maps || !p) return tw_set_error(ctx, TW_ERR_ARG, "null argument");
	if (xsize <= 0 || ysize <= 0 || ntiles == 0) return tw_set_error(ctx, TW_ERR_ARG, "empty heightmap");
	if (num_iters == 0 || p->erode_amount <= 0.0) {ctx->last_erosion_steps = 0; return TW_OK;} // src/erosion.cpp:16
	float *d_maps;
	tw_stage st(ctx);
	st.inout(&d_maps, maps, (size_t)xsize*ysize*ntiles*sizeof(float));
	rc = st.commit(); if (rc) return rc;
	float *d_minz = nullptr;
	if (min_zvals) {
		rc = tw_reserve(ctx, 2, OFF_TILES + (size_t)ntiles*sizeof(float)); if (rc) return rc;
		d_minz = (float *)((char *)ctx->d_scratch[2] + OFF_TILES);
		TW_CUDA(ctx, cudaMemcpyAsync(d_minz, min_zvals, (size_t)ntiles*sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
		TW_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	}
	rc = twi_erode(ctx, d_maps, ntiles, xsize, ysize, d_minz, min_zval_all, num_iters, p);
	if (rc) return rc;
	return st.finish();
}

int tw_create_zvals_batch(tw_ctx *ctx, const int32_t *origins_xy, uint32_t ntiles, int mesh_x_size, int mesh_y_size, float dx, float dy,
                          uint32_t zvsize, const tw_height_params *p, uint32_t erosion_iters, const tw_erosion_params *ep, float min_zval,
                          float *out, tw_minmax *mm)
{
	int rc = tw_enter(ctx); if (rc) return rc;
	if (!origins_xy || ntiles == 0 || !p || !out) return tw_set_error(ctx, TW_ERR_ARG, "null/empty argument");
	bool const erode = (erosion_iters > 0 && ep && ep->erode_amount > 0.0);
	ctx->last_erosion_steps = 0;
	if (!erode) {return tw_heightgen_tiles(ctx, origins_xy, ntiles, mesh_x_size, mesh_y_size, dx, dy, zvsize, p, out, mm);}
	tw_grid2d g; g.x0 = 0; g.y0 = 0; g.dx = dx; g.dy = dy; g.nx = zvsize; g.ny = zvsize;
	rc = validate_height(ctx, &g, p, out); if (rc) return rc;
	size_t const tile_elems = (size_t)zvsize*zvsize, n = tile_elems*ntiles;
	float *d_out;
	tw_stage st(ctx);
	if (p->gen_mode == TW_MGEN_SINE) { // sine tables live in the same scratch slot as the padded maps: no overlap, plain sequence
		st.out(&d_out, out, n*sizeof(float));
		rc = st.commit(); if (rc) return rc;
		rc = tw_heightgen_tiles(ctx, origins_xy, ntiles, mesh_x_size, mesh_y_size, dx, dy, zvsize, p, d_out, nullptr); if (rc) return rc;
		rc = tw_erode_tiles(ctx, d_out, ntiles, (int)zvsize, (int)zvsize, nullptr, min_zval, erosion_iters, ep); if (rc) return rc;
		if (mm) {for (uint32_t t = 0; t < ntiles; ++t) {rc = tw_minmax_f32(ctx, d_out + (size_t)t*tile_elems, tile_elems, mm + t); if (rc) return rc;}}
		return st.finish();
	}
	rc = twi_ensure_aux_streams(ctx); if (rc) return rc;
	bool const host_out = st.view(&d_out, out, n*sizeof(float));
	rc = st.commit(); if (rc) return rc;
	// The pipeline. Work per tile is heavy-tailed (ocean tiles: 1000 droplets x 1 move; mountain tiles: 1e5 moves in one serial chain), and a chain
	// cannot be sped up (csrc/tw_erosion.cu, plan_heavy), so the chains must START EARLY: (1) a coarse pre-pass evaluates the height function on an
	// 8x8 sample of every tile (4 M evaluations for 65536 tiles, < 1 ms) and counts the samples above the ocean-stop level - the same predictor the
	// erosion schedule uses, on 64 instead of 70756 cells; (2) the tiles are sorted heaviest first; (3) generation and erosion run chunk by chunk in
	// THAT order: generation of chunk k+1 (main stream) overlaps the droplet walks of chunks <= k (three high-priority streams; chunk 0, which holds
	// every long chain, has one to itself), so the long chains run under the generation of everything else and the last chunk to finish is the
	// lightest one. Tiles are generated / eroded in schedule order but stored at their caller-visible index (tile_perm). TW_PIPE_CHUNKS overrides
	// the chunk count (1 = the plain sequence); small batches use one chunk.
	size_t free_b = 0, total_b = 0;
	TW_CUDA(ctx, cudaMemGetInfo(&free_b, &total_b));
	size_t budget = (free_b + ctx->scratch_bytes[1])/3/3;
	if (budget < ((size_t)512 << 20)) budget = (size_t)512 << 20;
	// measured on B200 (tools/bench_pipeline_chunks.py, profiles/pipeline_chunks_r02.txt), 258^2 tiles, 1000 droplets: 8192 tiles 0.144 / 0.132 / 0.126 / 0.120 /
	// 0.128 / 0.179 s with 1 / 2 / 3 / 4 / 8 / 16 chunks (heaviest-first; in index order 4 chunks take 0.173 s); 65536 tiles 0.780 / 0.780 / 0.833 / 0.835 s with
	// 1 / 2 / 3 / 4: when the batch saturates the machine anyway, generation and erosion compete for the same issue slots and extra chunks only add overhead
	uint32_t want_chunks = (ntiles < 4096) ? 1 : ((ntiles <= 24576) ? 4 : 2);
	if (const char *e = getenv("TW_PIPE_CHUNKS")) {int const v = atoi(e); if (v >= 1 && v <= 64) want_chunks = (uint32_t)v;}
	uint32_t chunk = (ntiles + want_chunks - 1)/want_chunks;
	uint32_t const cap = twi_erode_chunk_for(budget, chunk, (int)zvsize, (int)zvsize);
	uint32_t const nchunks = (ntiles + cap - 1)/cap;
	chunk = (ntiles + nchunks - 1)/nchunks; // balanced
	bool const reorder = (nchunks > 1 && !getenv("TW_PIPE_NO_REORDER"));
	int const nes = (nchunks > 2) ? 3 : (int)nchunks; // erosion streams / scratch buffers
	size_t const sbytes = tw_align256(twi_erode_scratch_bytes(chunk, (int)zvsize, (int)zvsize));
	rc = tw_reserve(ctx, 1, sbytes*nes); if (rc) return rc;
	// slot 2: [small scalars | per-tile min/max | origins | sorted origins | work | order | hist(256) | coarse samples]
	uint32_t const CS = 8, cstep = (zvsize >= CS) ? zvsize/CS : 1;
	size_t const mm_bytes = tw_align256((size_t)ntiles*2*sizeof(unsigned)), org_bytes = tw_align256((size_t)ntiles*sizeof(float2));
	size_t const u_bytes = tw_align256((size_t)ntiles*sizeof(unsigned)), coarse_bytes = reorder ? tw_align256((size_t)ntiles*CS*CS*sizeof(float)) : 0;
	rc = tw_reserve(ctx, 2, OFF_TILES + mm_bytes + 2*org_bytes + 2*u_bytes + 1024 + coarse_bytes); if (rc) return rc;
	char *s2 = (char *)ctx->d_scratch[2] + OFF_TILES;
	unsigned *d_mm = (unsigned *)s2; s2 += mm_bytes;
	float2 *d_org = (float2 *)s2; s2 += org_bytes;
	float2 *d_org_sorted = (float2 *)s2; s2 += org_bytes;
	unsigned *d_work = (unsigned *)s2; s2 += u_bytes;
	unsigned *d_order = (unsigned *)s2; s2 += u_bytes;
	unsigned *d_hist = (unsigned *)s2; s2 += 1024;
	float *d_coarse = (float *)s2;
	unsigned long long *d_steps = (unsigned long long *)((char *)ctx->d_scratch[2] + 2048);
	{
		std::vector<float2> const org = tile_origins(origins_xy, ntiles, mesh_x_size, mesh_y_size, dx, dy);
		TW_CUDA(ctx, cudaMemcpyAsync(d_org, org.data(), (size_t)ntiles*sizeof(float2), cudaMemcpyHostToDevice, ctx->stream));
		TW_CUDA(ctx, cudaMemsetAsync(d_steps, 0, sizeof(unsigned long long), ctx->stream));
		TW_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); // org is a local vector; the aux streams must also see d_steps zeroed
	}
	const float2 *d_gen_org = d_org;
	const unsigned *d_perm = nullptr;
	if (reorder) { // (1) + (2): coarse estimate, heaviest-first order of the WHOLE batch
		tw_grid2d gc = g; gc.dx = dx*(float)cstep; gc.dy = dy*(float)cstep; gc.nx = CS; gc.ny = CS;
		for (uint32_t t0 = 0; t0 < ntiles; t0 += 65535) {
			uint32_t const nt = (ntiles - t0 < 65535) ? ntiles - t0 : 65535;
			rc = twi_heightgen(ctx, &gc, p, 1, 0, d_org + t0, nt, d_coarse + (size_t)t0*CS*CS, nullptr); if (rc) return rc;
		}
		rc = twi_coarse_work(ctx, d_coarse, CS*CS, ntiles, ep->water_plane_z - ep->half_dxy, d_work); if (rc) return rc;
		TW_CUDA(ctx, cudaMemsetAsync(d_hist, 0, 1024, ctx->stream));
		rc = twi_order_by_work(ctx, ctx->stream, d_work, ntiles, CS*CS, d_hist, d_order); if (rc) return rc;
		rc = twi_gather_origins(ctx, d_org, d_order, ntiles, d_org_sorted); if (rc) return rc;
		d_gen_org = d_org_sorted; d_perm = d_order;
	}
	std::vector<cudaEvent_t> ev(nchunks, nullptr);
	int status = TW_OK;
	for (uint32_t k = 0; k < nchunks && status == TW_OK; ++k) {
		uint32_t const t0 = k*chunk, nt = (ntiles - t0 < chunk) ? (ntiles - t0) : chunk;
		// schedule slots [t0, t0 + nt): with a permutation every kernel addresses `d_out` through it; without, the chunk is a contiguous slice
		float *maps = d_perm ? d_out : d_out + (size_t)t0*tile_elems;
		const unsigned *perm_k = d_perm ? d_perm + t0 : nullptr;
		ctx->tile_perm = perm_k;
		status = twi_heightgen(ctx, &g, p, 1, 0, d_gen_org + t0, nt, maps, nullptr);           // generation on ctx->stream
		ctx->tile_perm = nullptr;
		if (status) break;
		if (cudaEventCreateWithFlags(&ev[k], cudaEventDisableTiming) != cudaSuccess || cudaEventRecord(ev[k], ctx->stream) != cudaSuccess) {status = tw_set_error(ctx, TW_ERR_CUDA, "event"); break;}
		int const lane = (nes < 3) ? (int)(k % nes) : ((k == 0) ? 0 : 1 + (int)((k - 1) & 1)); // the heaviest chunk keeps a stream (and a scratch buffer) to itself
		cudaStream_t const es = ctx->aux_stream[lane];
		if (cudaStreamWaitEvent(es, ev[k], 0) != cudaSuccess) {status = tw_set_error(ctx, TW_ERR_CUDA, "cudaStreamWaitEvent"); break;}
		status = twi_erode_enqueue(ctx, es, 1 + lane, (char *)ctx->d_scratch[1] + (size_t)lane*sbytes, chunk, maps, nt, (int)zvsize, (int)zvsize, nullptr, min_zval, erosion_iters, ep, d_steps, perm_k);
		if (status) break;
		if (mm) {status = twi_minmax_tiles(ctx, es, maps, tile_elems, nt, d_perm ? d_mm : d_mm + 2*(size_t)t0, perm_k); if (status) break;}
		if (host_out && !d_perm && cudaMemcpyAsync(out + (size_t)t0*tile_elems, maps, (size_t)nt*tile_elems*sizeof(float), cudaMemcpyDeviceToHost, es) != cudaSuccess) {status = tw_set_error(ctx, TW_ERR_CUDA, "D2H");}
	}
	cudaError_t e0 = cudaStreamSynchronize(ctx->stream), e1 = cudaStreamSynchronize(ctx->aux_stream[0]), e2 = cudaStreamSynchronize(ctx->aux_stream[1]), e3 = cudaStreamSynchronize(ctx->aux_stream[2]);
	for (cudaEvent_t e : ev) {if (e) cudaEventDestroy(e);}
	if (status) return status;
	if (e0 != cudaSuccess || e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) return tw_set_error(ctx, TW_ERR_CUDA, "tile pipeline: %s", cudaGetErrorString(e0 != cudaSuccess ? e0 : (e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3))));
	if (host_out && d_perm) {TW_CUDA(ctx, cudaMemcpy(out, d_out, n*sizeof(float), cudaMemcpyDeviceToHost));} // schedule order scatters a chunk over the whole buffer: one copy at the end
	unsigned long long h_steps = 0;
	TW_CUDA(ctx, cudaMemcpy(&h_steps, d_steps, sizeof(h_steps), cudaMemcpyDeviceToHost));
	ctx->last_erosion_steps = h_steps;
	if (mm) {rc = read_minmax(ctx, d_mm, mm, ntiles); if (rc) return rc;}
	return TW_OK;
}

int tw_heightmap_sample_tiles(tw_ctx *ctx, const uint8_t *data16, const tw_hmap_sampler *hs, const int32_t *origins_xy, uint32_t ntiles, uint32_t zvsize, float *out) {
	int rc = tw_enter(ctx); if (rc) return rc;
	if (!data16 || !hs || !origins_xy || !out || ntiles == 0 || zvsize == 0) return tw_set_error(ctx, TW_ERR_ARG, "null/empty argument");
	if (hs->width <= 0 || hs->height <= 0 || hs->edge_mode < 0 || hs->edge_mode > 2) return tw_set_error(ctx, TW_ERR_ARG, "bad heightmap sampler");
	if (ntiles > 65535) return tw_set_error(ctx, TW_ERR_ARG, "at most 65535 tiles per call");
	int32_t *d_org; const uint8_t *d_img; float *d_out;
	tw_stage st(ctx);
	st.temp(&d_org, (size_t)ntiles*8); // origins_xy is a host array
	st.in(&d_img, data16, (size_t)2*hs->width*hs->height);
	st.out(&d_out, out, (size_t)ntiles*zvsize*zvsize*sizeof(float));
	rc = st.commit(); if (rc) return rc;
	TW_CUDA(ctx, cudaMemcpyAsync(d_org, origins_xy, (size_t)ntiles*8, cudaMemcpyHostToDevice, ctx->stream));
	rc = twi_hmap_sample_tiles(ctx, d_img, hs, d_org, ntiles, zvsize, d_out); if (rc) return rc;
	return st.finish(); // also waits for the read of origins_xy, the caller's buffer
}

// ------------------------------------------------------------------------------------------------ per-tile normals and ambient occlusion (N1)
int tw_tile_normals_batch(tw_ctx *ctx, const float *zvals, uint32_t ntiles, uint32_t zvsize, float dx_val, float dy_val, uint8_t *rgba, float *min_normal_z) {
	int rc = tw_enter(ctx); if (rc) return rc;
	if (!zvals || !rgba || ntiles == 0 || zvsize < 2) return tw_set_error(ctx, TW_ERR_ARG, "null/empty argument");
	if (ntiles > 65535) return tw_set_error(ctx, TW_ERR_ARG, "at most 65535 tiles per call");
	size_t const stride = zvsize - 1;
	unsigned *d_mn; const float *d_z; uint8_t *d_rgba;
	tw_stage st(ctx);
	st.temp(&d_mn, (size_t)ntiles*sizeof(unsigned));
	st.in(&d_z, zvals, (size_t)ntiles*zvsize*zvsize*sizeof(float));
	st.out(&d_rgba, rgba, (size_t)ntiles*stride*stride*4);
	rc = st.commit(); if (rc) return rc;
	{
		std::vector<unsigned> init(ntiles, tw_f2ord(1.0f)); // min_normal_z = 1.0, src/tiled_mesh.cpp:868
		TW_CUDA(ctx, cudaMemcpyAsync(d_mn, init.data(), ntiles*sizeof(unsigned), cudaMemcpyHostToDevice, ctx->stream));
		TW_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	}
	rc = twi_tile_normals(ctx, d_z, ntiles, zvsize, dx_val, dy_val, d_rgba, d_mn); if (rc) return rc;
	std::vector<unsigned> mn(ntiles);
	if (min_normal_z) {TW_CUDA(ctx, cudaMemcpyAsync(mn.data(), d_mn, ntiles*sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream));}
	rc = st.finish(); if (rc) return rc;
	if (min_normal_z) {for (uint32_t t = 0; t < ntiles; ++t) {min_normal_z[t] = tw_ord2f(mn[t]);}}
	return TW_OK;
}

// context grids of `nt` tiles at (x1 - AO_RAY_LEN, y1 - AO_RAY_LEN) into d_cz; skip_inside: leave the zvsize^2 interior unwritten (never read)
static int gen_ao_contexts(tw_ctx *ctx, const int32_t *origins_xy, uint32_t nt, int mesh_x_size, int mesh_y_size, float dx, float dy, uint32_t zvsize,
                           const tw_height_params *p, bool skip_inside, std::vector<int32_t> &org, float *d_cz)
{
	uint32_t const ray = 36, csz = zvsize - 1 + 2*ray; // AO_RAY_LEN, context_sz (src/tiled_mesh.cpp:43,601)
	for (uint32_t t = 0; t < nt; ++t) {org[2*t] = origins_xy[2*t] - (int32_t)ray; org[2*t + 1] = origins_xy[2*t + 1] - (int32_t)ray;}
	if (skip_inside) {ctx->skip_rect[0] = ctx->skip_rect[1] = ray; ctx->skip_rect[2] = ctx->skip_rect[3] = zvsize;}
	int const rc = tw_heightgen_tiles(ctx, org.data(), nt, mesh_x_size, mesh_y_size, dx, dy, csz, p, d_cz, nullptr); // device output: stages nothing in the caller's slot 0
	ctx->skip_rect[0] = ctx->skip_rect[1] = ctx->skip_rect[2] = ctx->skip_rect[3] = 0;
	return rc;
}

int tw_tile_ao_batch(tw_ctx *ctx, const float *zvals, const int32_t *origins_xy, uint32_t ntiles, int mesh_x_size, int mesh_y_size,
                     float dx, float dy, uint32_t zvsize, const tw_height_params *p, float half_dxy, uint8_t *ao)
{
	int rc = tw_enter(ctx); if (rc) return rc;
	if (!zvals || !origins_xy || !p || !ao || ntiles == 0 || zvsize < 2) return tw_set_error(ctx, TW_ERR_ARG, "null/empty argument");
	uint32_t const ray = 36, stride = zvsize - 1, csz = stride + 2*ray; // AO_RAY_LEN, context_sz (src/tiled_mesh.cpp:43,601)
	size_t const tile_elems = (size_t)zvsize*zvsize, ctx_elems = (size_t)csz*csz, ao_elems = (size_t)stride*stride;
	bool const ctx_inside = (p->gen_mode >= TW_MGEN_SIMPLEX_GPU); // use_ao_zvals: the rays test the un-eroded context inside the tile too (src/tiled_mesh.cpp:604)
	// chunk of tiles whose context grids fit in ~2 GB
	uint32_t chunk = (uint32_t)std::min<size_t>(ntiles, std::max<size_t>(1, ((size_t)2 << 30)/(ctx_elems*sizeof(float))));
	if (chunk > 65535) chunk = 65535;
	const float *z_buf; uint8_t *ao_buf; float *d_cz; // host zvals / ao: one chunk's region, device ones: the whole buffer
	tw_stage st(ctx);
	bool const host_z = st.view(&z_buf, zvals, (size_t)chunk*tile_elems*sizeof(float));
	st.temp(&d_cz, (size_t)chunk*ctx_elems*sizeof(float));
	bool const host_ao = st.view(&ao_buf, ao, (size_t)chunk*ao_elems);
	rc = st.commit(); if (rc) return rc;
	std::vector<int32_t> org(2*(size_t)chunk);
	for (uint32_t t0 = 0; t0 < ntiles; t0 += chunk) {
		uint32_t const nt = (ntiles - t0 < chunk) ? ntiles - t0 : chunk;
		const float *d_z = host_z ? z_buf : zvals + (size_t)t0*tile_elems;
		uint8_t *d_ao = host_ao ? ao_buf : ao + (size_t)t0*ao_elems;
		if (host_z) {TW_CUDA(ctx, cudaMemcpyAsync(const_cast<float *>(z_buf), zvals + (size_t)t0*tile_elems, (size_t)nt*tile_elems*sizeof(float), cudaMemcpyHostToDevice, ctx->stream));}
		rc = gen_ao_contexts(ctx, origins_xy + 2*(size_t)t0, nt, mesh_x_size, mesh_y_size, dx, dy, zvsize, p, !ctx_inside, org, d_cz);
		if (rc) return rc;
		rc = twi_tile_ao(ctx, d_z, d_cz, nt, zvsize, half_dxy, ctx_inside, d_ao); if (rc) return rc;
		if (host_ao) {TW_CUDA(ctx, cudaMemcpyAsync(ao + (size_t)t0*ao_elems, d_ao, (size_t)nt*ao_elems, cudaMemcpyDeviceToHost, ctx->stream));}
		TW_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	}
	return TW_OK;
}

int tw_create_zvals_ao_batch(tw_ctx *ctx, const int32_t *origins_xy, uint32_t ntiles, int mesh_x_size, int mesh_y_size, float dx, float dy,
                             uint32_t zvsize, const tw_height_params *p, uint32_t erosion_iters, const tw_erosion_params *ep, float min_zval,
                             float half_dxy, float *zvals, uint8_t *ao, tw_minmax *mm)
{
	int rc = tw_enter(ctx); if (rc) return rc;
	if (!origins_xy || !p || !zvals || !ao || ntiles == 0 || zvsize < 2) return tw_set_error(ctx, TW_ERR_ARG, "null/empty argument");
	uint32_t const ray = 36, stride = zvsize - 1, csz = stride + 2*ray;
	size_t const tile_elems = (size_t)zvsize*zvsize, ctx_elems = (size_t)csz*csz, ao_elems = (size_t)stride*stride;
	bool const ctx_mode = (p->gen_mode >= TW_MGEN_SIMPLEX_GPU); // one generation, zvals cut from the context (src/tiled_mesh.cpp:479-487,505)
	bool const erode = (erosion_iters > 0 && ep && ep->erode_amount > 0.0);
	uint32_t chunk = (uint32_t)std::min<size_t>(ntiles, std::max<size_t>(1, ((size_t)2 << 30)/(ctx_elems*sizeof(float))));
	if (chunk > 65535) chunk = 65535;
	float *d_cz, *z_buf; unsigned *d_mm; uint8_t *ao_buf; // host zvals / ao: one chunk's region, device ones: the whole buffer
	tw_stage st(ctx);
	st.temp(&d_cz, (size_t)chunk*ctx_elems*sizeof(float));
	st.temp(&d_mm, (size_t)chunk*2*sizeof(unsigned));
	bool const host_z = st.view(&z_buf, zvals, (size_t)chunk*tile_elems*sizeof(float));
	bool const host_ao = st.view(&ao_buf, ao, (size_t)chunk*ao_elems);
	rc = st.commit(); if (rc) return rc;
	std::vector<int32_t> org(2*(size_t)chunk);
	uint64_t moves = 0;
	for (uint32_t t0 = 0; t0 < ntiles; t0 += chunk) {
		uint32_t const nt = (ntiles - t0 < chunk) ? ntiles - t0 : chunk;
		const int32_t *orgs = origins_xy + 2*(size_t)t0;
		float *d_z = host_z ? z_buf : zvals + (size_t)t0*tile_elems;
		uint8_t *d_ao = host_ao ? ao_buf : ao + (size_t)t0*ao_elems;
		if (ctx_mode) {
			rc = gen_ao_contexts(ctx, orgs, nt, mesh_x_size, mesh_y_size, dx, dy, zvsize, p, false, org, d_cz); if (rc) return rc;
			rc = twi_tile_cut(ctx, d_cz, nt, zvsize, d_z); if (rc) return rc;
		}
		else {rc = tw_heightgen_tiles(ctx, orgs, nt, mesh_x_size, mesh_y_size, dx, dy, zvsize, p, d_z, nullptr); if (rc) return rc;}
		if (erode) {
			rc = tw_erode_tiles(ctx, d_z, nt, (int)zvsize, (int)zvsize, nullptr, min_zval, erosion_iters, ep); if (rc) return rc; // tile_t::create_zvals: apply_erosion(zvals, ..., zmin, ...)
			moves += ctx->last_erosion_steps;
		}
		if (!ctx_mode) {rc = gen_ao_contexts(ctx, orgs, nt, mesh_x_size, mesh_y_size, dx, dy, zvsize, p, true, org, d_cz); if (rc) return rc;}
		rc = twi_tile_ao(ctx, d_z, d_cz, nt, zvsize, half_dxy, ctx_mode, d_ao); if (rc) return rc;
		if (mm) {
			rc = twi_init_minmax(ctx, d_mm, nt); if (rc) return rc;
			rc = twi_minmax_tiles(ctx, ctx->stream, d_z, tile_elems, nt, d_mm); if (rc) return rc;
		}
		if (host_z)  {TW_CUDA(ctx, cudaMemcpyAsync(zvals + (size_t)t0*tile_elems, d_z, (size_t)nt*tile_elems*sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));}
		if (host_ao) {TW_CUDA(ctx, cudaMemcpyAsync(ao + (size_t)t0*ao_elems, d_ao, (size_t)nt*ao_elems, cudaMemcpyDeviceToHost, ctx->stream));}
		if (mm) {rc = read_minmax(ctx, d_mm, mm + t0, nt); if (rc) return rc;}
		TW_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
	}
	ctx->last_erosion_steps = moves;
	return TW_OK;
}

// ------------------------------------------------------------------------------------------------ point queries
int tw_eval_points(tw_ctx *ctx, const float *xy, size_t n, const tw_height_params *p, const tw_point_query *q, float *out) {
	int rc = tw_enter(ctx); if (rc) return rc;
	if (!xy || !p || !q || !out) return tw_set_error(ctx, TW_ERR_ARG, "null argument");
	if (n == 0) return TW_OK;
	if (!ctx->have_sin) return tw_set_error(ctx, TW_ERR_STATE, "tw_set_sin_table() has not been called");
	const float *d_xy; float *d_out;
	tw_stage st(ctx);
	st.in(&d_xy, xy, 2*n*sizeof(float));
	st.out(&d_out, out, n*sizeof(float));
	rc = st.commit(); if (rc) return rc;
	rc = twi_eval_points(ctx, d_xy, n, p, q, d_out); if (rc) return rc;
	return st.finish();
}

int tw_erode(tw_ctx *ctx, float *heightmap, int xsize, int ysize, float min_zval, uint32_t num_iters, const tw_erosion_params *p) {
	return tw_erode_tiles(ctx, heightmap, 1, xsize, ysize, nullptr, min_zval, num_iters, p);
}

int tw_erode_parallel(tw_ctx *ctx, float *heightmap, int xsize, int ysize, float min_zval, uint32_t num_iters, const tw_erosion_params *p, uint32_t num_threads) {
	int rc = tw_enter(ctx); if (rc) return rc;
	if (!heightmap || !p) return tw_set_error(ctx, TW_ERR_ARG, "null argument");
	if (xsize <= 0 || ysize <= 0) return tw_set_error(ctx, TW_ERR_ARG, "empty heightmap");
	if (num_iters == 0 || p->erode_amount <= 0.0) {ctx->last_erosion_steps = 0; return TW_OK;} // src/erosion.cpp:16
	float *d_map;
	tw_stage st(ctx);
	st.inout(&d_map, heightmap, (size_t)xsize*ysize*sizeof(float));
	rc = st.commit(); if (rc) return rc;
	rc = twi_erode_parallel(ctx, d_map, xsize, ysize, min_zval, num_iters, p, num_threads); if (rc) return rc;
	return st.finish();
}

// ------------------------------------------------------------------------------------------------ voxels
int tw_voxel_fill(tw_ctx *ctx, const tw_voxel_params *vp, const float *rdata420, float *out) {
	int rc = tw_enter(ctx); if (rc) return rc;
	if (!vp || !out) return tw_set_error(ctx, TW_ERR_ARG, "null argument");
	if (!ctx->have_sin) return tw_set_error(ctx, TW_ERR_STATE, "tw_set_sin_table() has not been called");
	if (vp->gen_mode < 0 || vp->gen_mode > TW_MGEN_DWARP_GPU) return tw_set_error(ctx, TW_ERR_ARG, "bad gen_mode");
	float *d_out;
	tw_stage st(ctx);
	st.out(&d_out, out, (size_t)vp->nx*vp->ny*vp->nz*sizeof(float));
	rc = st.commit(); if (rc) return rc;
	rc = twi_voxel_fill(ctx, vp, rdata420, d_out); if (rc) return rc;
	return st.finish();
}

// ------------------------------------------------------------------------------------------------ streaming passes
int tw_heightmap_from_floats_u16(tw_ctx *ctx, const float *vals, size_t n, float val_mult, float val_add, uint8_t *out2n) {
	int rc = tw_enter(ctx); if (rc) return rc;
	if (!vals || !out2n || n == 0) return tw_set_error(ctx, TW_ERR_ARG, "null/empty argument");
	const float *d_in; uint8_t *d_out;
	tw_stage st(ctx);
	st.in(&d_in, vals, n*sizeof(float));
	st.out(&d_out, out2n, 2*n);
	rc = st.commit(); if (rc) return rc;
	rc = tw_reserve(ctx, 2, OFF_TILES); if (rc) return rc;
	unsigned *d_bad = (unsigned *)((char *)ctx->d_scratch[2] + OFF_BAD);
	TW_CUDA(ctx, cudaMemsetAsync(d_bad, 0, sizeof(unsigned), ctx->stream));
	rc = twi_from_floats_u16(ctx, d_in, n, val_mult, val_add, d_out, d_bad);
	if (rc) return rc;
	unsigned bad = 0;
	TW_CUDA(ctx, cudaMemcpyAsync(&bad, d_bad, sizeof(bad), cudaMemcpyDeviceToHost, ctx->stream));
	rc = st.finish(); if (rc) return rc;
	if (bad) return tw_set_error(ctx, TW_ERR_ARG, "from_floats: value outside [0,256) (the reference asserts, src/heightmap.cpp:211)");
	return TW_OK;
}

int tw_heightmap_to_floats_u16(tw_ctx *ctx, const uint8_t *data2n, size_t n, float val_mult, float val_add, float *vals) {
	int rc = tw_enter(ctx); if (rc) return rc;
	if (!vals || !data2n || n == 0) return tw_set_error(ctx, TW_ERR_ARG, "null/empty argument");
	const uint8_t *d_in; float *d_out;
	tw_stage st(ctx);
	st.in(&d_in, data2n, 2*n);
	st.out(&d_out, vals, n*sizeof(float));
	rc = st.commit(); if (rc) return rc;
	rc = twi_to_floats_u16(ctx, d_in, n, val_mult, val_add, d_out); if (rc) return rc;
	return st.finish();
}

int tw_proc_gen_heightmap(tw_ctx *ctx, uint32_t width, uint32_t height, float dx_val, float dy_val, const tw_height_params *p,
                          uint32_t erosion_iters, const tw_erosion_params *ep, uint8_t *data16, float *vals, tw_heightmap_info *info)
{
	int rc = tw_enter(ctx); if (rc) return rc;
	if (!p || !data16 || width == 0 || height == 0) return tw_set_error(ctx, TW_ERR_ARG, "null/empty argument");
	tw_grid2d g; g.x0 = -0.5*width; g.y0 = -0.5*height; g.dx = dx_val; g.dy = dy_val; g.nx = width; g.ny = height; // src/heightmap.cpp:135
	size_t const n = (size_t)width*height;
	float *d_vals; uint8_t *d_img;
	tw_stage st(ctx);
	if (vals) {st.out(&d_vals, vals, n*sizeof(float));} else {st.temp(&d_vals, n*sizeof(float));}
	st.out(&d_img, data16, 2*n);
	rc = st.commit(); if (rc) return rc;
	rc = validate_height(ctx, &g, p, d_vals); if (rc) return rc;
	unsigned *d_mm;
	tw_minmax mm;
	rc = single_minmax(ctx, &d_mm); if (rc) return rc;
	rc = twi_heightgen(ctx, &g, p, 1, 0, nullptr, 1, d_vals, d_mm); if (rc) return rc;
	rc = read_minmax(ctx, d_mm, &mm, 1); if (rc) return rc;
	uint64_t moves = 0;
	if (erosion_iters > 0 && ep && ep->erode_amount > 0.0) { // run_erosion: min_zval = min over vals (src/heightmap.cpp:155-156)
		rc = twi_erode(ctx, d_vals, 1, (int)width, (int)height, nullptr, mm.zmin, erosion_iters, ep); if (rc) return rc;
		moves = ctx->last_erosion_steps;
		rc = twi_init_minmax(ctx, d_mm, 1); if (rc) return rc;
		rc = twi_minmax(ctx, d_vals, n, d_mm); if (rc) return rc;
		rc = read_minmax(ctx, d_mm, &mm, 1); if (rc) return rc; // get_heightmap_z_range
	}
	float const min_z = mm.zmin, max_z = mm.zmax;
	float const TOLERANCE = 1.0E-12, READ_MESH_H_SCALE = 0.0008; // src/3DWorld.h:50, src/mesh_gen.cpp:22
	float const dzr = max_z - min_z, dz = (TOLERANCE < dzr) ? dzr : TOLERANCE; // max(TOLERANCE, (max_z - min_z))
	float const dz255 = dz/255.0;                                             // set_mesh_height_scales_for_zval_range(min_z, dz/255.0)
	float const mesh_file_scale = dz255/(READ_MESH_H_SCALE*p->mesh_height_scale*p->mesh_scale_z_inv);
	float const mesh_file_tz    = min_z/p->mesh_scale_z_inv;
	float const val_mult = READ_MESH_H_SCALE*p->mesh_height_scale*mesh_file_scale*p->mesh_scale_z_inv; // get_mh_texture_mult()
	float const val_add  = mesh_file_tz*p->mesh_scale_z_inv;                                             // get_mh_texture_add()
	unsigned *d_bad = (unsigned *)((char *)ctx->d_scratch[2] + OFF_BAD);
	TW_CUDA(ctx, cudaMemsetAsync(d_bad, 0, sizeof(unsigned), ctx->stream));
	rc = twi_from_floats_u16(ctx, d_vals, n, val_mult, val_add, d_img, d_bad); if (rc) return rc;
	unsigned bad = 0;
	TW_CUDA(ctx, cudaMemcpyAsync(&bad, d_bad, sizeof(bad), cudaMemcpyDeviceToHost, ctx->stream));
	rc = st.finish(); if (rc) return rc;
	ctx->last_erosion_steps = moves;
	if (info) {info->min_z = min_z; info->max_z = max_z; info->val_mult = val_mult; info->val_add = val_add; info->mesh_file_scale = mesh_file_scale; info->mesh_file_tz = mesh_file_tz; info->erosion_moves = moves;}
	if (bad) return tw_set_error(ctx, TW_ERR_ARG, "from_floats: value outside [0,256) (the reference asserts, src/heightmap.cpp:211)");
	return TW_OK;
}

int tw_minmax_f32(tw_ctx *ctx, const float *vals, size_t n, tw_minmax *mm) {
	int rc = tw_enter(ctx); if (rc) return rc;
	if (!vals || !mm || n == 0) return tw_set_error(ctx, TW_ERR_ARG, "null/empty argument");
	const float *d_in;
	tw_stage st(ctx);
	st.in(&d_in, vals, n*sizeof(float));
	rc = st.commit(); if (rc) return rc;
	unsigned *d_mm;
	rc = single_minmax(ctx, &d_mm); if (rc) return rc;
	rc = twi_minmax(ctx, d_in, n, d_mm); if (rc) return rc;
	return read_minmax(ctx, d_mm, mm, 1);
}

} // extern "C"
