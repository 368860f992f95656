// tw_internal.h - context object and helpers shared by the CUDA translation units of lib3dworld_b200.so
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <stdio.h>
#include <string.h>
#include "../../include/tw3d.h"

struct tw_async_state {
	bool pending = false;
	cudaEvent_t done = nullptr;
	float *host_out = nullptr;      // user host buffer (nullptr => result stays on device)
	tw_minmax *host_mm = nullptr;
	uint32_t n_mm = 0;
};

struct tw_ctx {
	int device = 0;
	cudaStream_t stream = nullptr;
	cudaStream_t aux_stream[3] = {nullptr, nullptr, nullptr}; // erosion side of the fused tile pipeline (tw_create_zvals_batch): [0] the heaviest chunk, [1]/[2] alternate
	cudaStream_t heavy_stream[4] = {nullptr, nullptr, nullptr, nullptr}; // fork/join streams of the erosion's latency-mode launch (lane 0: ctx->stream, 1..3: aux_stream[0..2])
	cudaEvent_t  ev_fork[4] = {nullptr, nullptr, nullptr, nullptr}, ev_join[4] = {nullptr, nullptr, nullptr, nullptr};
	const unsigned *tile_perm = nullptr; // set around twi_heightgen by the tile pipeline: output slot of each generated tile
	char err[512] = {0};
	uint64_t launches = 0;
	uint64_t last_erosion_steps = 0;
	// uploaded tables
	float  *d_sin_table = nullptr;     // [65536]  sin_table (src/sinf.h:11)
	void   *d_glm3_lut = nullptr;      // float4[2*291]: simplex(vec3) / perlin(vec3) normalised gradient + permute tables (voxel density)
	void   *d_simplex_lut = nullptr;   // float4[291] {a0, h, norm, permute(k)}: simplex hash/gradient table (tw_noise2.cuh), built on first use
	float2 *d_dir_table = nullptr;     // [1000000] (cosf(a_k), sinf(a_k)), a_k = float(1e-6*k)*TWO_PI, host libm (src/erosion.cpp:85-86)
	float  *d_sine_params = nullptr;   // [450] sinTable
	float   h_sine_params[TW_F_TABLE_SIZE*5];
	bool have_sin = false, have_sine_params = false;
	// growable device scratch
	void  *d_scratch[3] = {nullptr, nullptr, nullptr}; // 0: caller-buffer staging (tw_stage only), 1: tables / padded heightmaps, 2: small (minmax, counters, origins)
	size_t scratch_bytes[3] = {0, 0, 0};
	bool scratch0_held = false;  // a tw_stage of the running entry point has buffers in slot 0: an entry it calls must not stage into slot 0
	// pinned host staging for small results
	void  *h_pinned = nullptr;
	size_t pinned_bytes = 0;
	tw_async_state async;
	void *dist = nullptr;        // tw_dist_state (tw_multi.cu): NCCL communicator of the one-process-per-GPU mode
	unsigned skip_rect[4] = {0, 0, 0, 0}; // x0, y0, w, h of the cells twi_heightgen's packed noise kernels leave unwritten (set around AO context generation only)
};

int  tw_set_error(tw_ctx *ctx, int status, const char *fmt, ...);
int  tw_reserve(tw_ctx *ctx, int slot, size_t bytes);           // grow d_scratch[slot]; returns TW_OK / TW_ERR_CUDA
int  tw_reserve_pinned(tw_ctx *ctx, size_t bytes);
bool tw_is_device_ptr(const void *p);
int  tw_enter(tw_ctx *ctx);  // first call of every entry point that works on ctx: selects ctx->device, completes a pending tw_heightgen_2d_launch

inline size_t tw_align256(size_t b) {return (b + 255) & ~(size_t)255;}

// Device views of one entry-point call's caller buffers, which include/tw3d.h lets be host or device memory. A device buffer (or null) is used in place;
// a host buffer, and every temp(), gets its own 256-byte-aligned region of scratch slot 0. Declare the buffers, then commit() reserves slot 0 once,
// assigns the device pointers and uploads in / inout; finish() downloads out / inout and synchronises ctx->stream. view() gives the region but leaves
// the copies to the call site (chunked, banded or pipelined transfers). slack: bytes the region has beyond the copied size (word atomics on a flag tail).
class tw_stage {
public:
	explicit tw_stage(tw_ctx *ctx) : ctx_(ctx) {}
	~tw_stage() {if (held_) ctx_->scratch0_held = false;}
	tw_stage(const tw_stage &) = delete;
	tw_stage &operator=(const tw_stage &) = delete;
	template<class T> void in   (const T **d, const T *caller, size_t bytes)        {add(d, caller, bytes, 0, IN);}
	template<class T> void out  (T **d, T *caller, size_t bytes, size_t slack = 0)  {add(d, caller, bytes, slack, OUT);}
	template<class T> void inout(T **d, T *caller, size_t bytes, size_t slack = 0)  {add(d, caller, bytes, slack, IN | OUT);}
	template<class T> bool view (T **d, T *caller, size_t bytes)                    {return add(d, caller, bytes, 0, 0);} // true: caller is host memory
	template<class T> void temp (T **d, size_t bytes)                               {add(d, nullptr, bytes, 0, TEMP);}
	int commit();
	int finish();
	static bool is_host(const void *p) {return p && !tw_is_device_ptr(p);}
private:
	enum {IN = 1, OUT = 2, TEMP = 4, MAX_BUFFERS = 8};
	struct entry {void *d; const void *caller; void *dev; size_t bytes, region; int dir; bool host;};
	bool add(void *d, const void *caller, size_t bytes, size_t slack, int dir);
	tw_ctx *ctx_;
	entry e_[MAX_BUFFERS];
	int n_ = 0;
	bool held_ = false;
};

#define TW_CUDA(ctx, call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { \
	return tw_set_error((ctx), TW_ERR_CUDA, "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); } } while (0)
#define TW_LAUNCH_CHECK(ctx) do { (ctx)->launches++; cudaError_t e_ = cudaGetLastError(); if (e_ != cudaSuccess) { \
	return tw_set_error((ctx), TW_ERR_CUDA, "%s:%d kernel launch: %s", __FILE__, __LINE__, cudaGetErrorString(e_)); } } while (0)

// ---- constants shared by host and device code (src/3DWorld.h:43,129; src/sinf.h:8-9) ----
#define TW_TSIZE 32768
constexpr float TW_PI_F     = 3.141592654f;
constexpr float TW_TWO_PI_F = (float)(2.0*TW_PI_F);
constexpr float TW_SSCALE   = (float)TW_TSIZE/TW_TWO_PI_F;

// float -> int conversion with the semantics the reference build gets from x86 cvttss2si: truncation toward zero, and the
// "integer indefinite" value INT_MIN for NaN and for anything outside int range (CUDA's cvt would give 0 / saturate instead).
// This matters: a droplet whose state went NaN (SURVEY.md section 7 "NaN hazard") terminates because (int)floor(NaN) == INT_MIN
// makes it "outside" (src/erosion.cpp:93,101), and SINF's table index (src/sinf.h:11) wraps the same way for huge arguments.
__device__ __forceinline__ int tw_x86_f2i(float f) {
	return (f >= -2147483648.0f && f < 2147483648.0f) ? __float2int_rz(f) : (int)0x80000000;
}

// order-preserving float <-> uint encoding for atomicMin/atomicMax reductions
__host__ __device__ inline unsigned tw_f2ord(float f) {
#ifdef __CUDA_ARCH__
	unsigned u = __float_as_uint(f);
#else
	unsigned u; memcpy(&u, &f, 4);
#endif
	return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ inline float tw_ord2f(unsigned u) {
	u = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
#ifdef __CUDA_ARCH__
	return __uint_as_float(u);
#else
	float f; memcpy(&f, &u, 4); return f;
#endif
}

// entry points implemented in the individual .cu files (called from tw_api.cu)
int twi_heightgen(tw_ctx *ctx, const tw_grid2d *g, const tw_height_params *p, int enable_glaciate, int min_start_sin,
                  const float2 *d_tile_origins, uint32_t ntiles, float *d_out, unsigned *d_mm_ord, float *h_out_bands = nullptr);
int twi_tile_weights(tw_ctx *ctx, const float *d_zvals, const float *d_rand, uint32_t ntiles, uint32_t zvsize, const float *d_tile_params, const tw_weight_params *W, uint8_t *d_out, uint8_t *d_flags);
int twi_heightgen_sine_tiles(tw_ctx *ctx, const tw_grid2d *g, const tw_height_params *p, int enable_glaciate, int min_start_sin, const float2 *h_org, uint32_t ntiles,
                             float *d_out, unsigned *d_mm_ord);
int twi_ensure_aux_streams(tw_ctx *ctx);
int twi_erode(tw_ctx *ctx, float *d_maps, uint32_t ntiles, int xsize, int ysize, const float *d_min_zvals, float min_zval_all,
              uint32_t num_iters, const tw_erosion_params *p);
int twi_hmap_sample_tiles(tw_ctx *ctx, const uint8_t *d_data16, const tw_hmap_sampler *hs, const void *d_origins, uint32_t ntiles, uint32_t zvsize, float *d_out);
int twi_tile_normals(tw_ctx *ctx, const float *d_zvals, uint32_t ntiles, uint32_t zvsize, float dx_val, float dy_val, unsigned char *d_rgba, unsigned *d_min_nz_ord);
int twi_tile_ao(tw_ctx *ctx, const float *d_zvals, const float *d_czv, uint32_t ntiles, uint32_t zvsize, float half_dxy, bool ctx_inside, unsigned char *d_ao);
int twi_tile_cut(tw_ctx *ctx, const float *d_czv, uint32_t ntiles, uint32_t zvsize, float *d_zvals);
int twi_eval_points(tw_ctx *ctx, const float *d_xy, size_t n, const tw_height_params *p, const tw_point_query *q, float *d_out);
int twi_erode_parallel(tw_ctx *ctx, float *d_map, int xsize, int ysize, float min_zval, uint32_t num_iters, const tw_erosion_params *p, uint32_t num_threads);
size_t   twi_erode_scratch_bytes(uint32_t chunk, int xsize, int ysize);
uint32_t twi_erode_chunk_for(size_t budget, uint32_t ntiles, int xsize, int ysize);
int twi_erode_enqueue(tw_ctx *ctx, cudaStream_t st, int lane, void *scratch, uint32_t capacity, float *maps, uint32_t nt, int xsize, int ysize,
                      const float *d_min_zvals, float min_zval_all, uint32_t num_iters, const tw_erosion_params *p, unsigned long long *d_steps,
                      const unsigned *d_perm = nullptr);
// coherent batched erosion (tw_erode_sweeps*): per-band building blocks, all enqueued on ctx->stream
int twi_sweep_pad(tw_ctx *ctx, const float *U, int u0, int xsize, int ysize, int E0, int rows, float *P);
int twi_sweep_view();
int twi_sweep_walk(tw_ctx *ctx, float *P, long long *D, int xsize, int ysize, int E0, int own0, int own1, int halo_rule, unsigned it0, unsigned it1,
                   const tw_erosion_params *p, unsigned long long *d_steps);
int twi_sweep_add(tw_ctx *ctx, long long *D, const long long *R, size_t n);
int twi_sweep_apply(tw_ctx *ctx, float *P, long long *D, size_t n);
int twi_sweep_unpad(tw_ctx *ctx, const float *P, int E0, int xsize, int y0, int y1, float min_zval, float *out);
int twi_tile_bounds(tw_ctx *ctx, const float *d_zvals, uint32_t ntiles, uint32_t zvsize, float wpz_max, void *d_sub);
int twi_glaciate_mesh(tw_ctx *ctx, float *d_mesh, int nx, int ny, int xoff2, int yoff2, int MX, int MY, const tw_height_params *p, unsigned *d_mm);
int twi_voxel_fill(tw_ctx *ctx, const tw_voxel_params *vp, const float *rdata420, float *d_out);
int twi_from_floats_u16(tw_ctx *ctx, const float *d_vals, size_t n, float val_mult, float val_add, uint8_t *d_out, unsigned *d_bad);
int twi_to_floats_u16(tw_ctx *ctx, const uint8_t *d_data, size_t n, float val_mult, float val_add, float *d_vals);
int twi_minmax(tw_ctx *ctx, const float *d_vals, size_t n, unsigned *d_mm_ord);
int twi_minmax_tiles(tw_ctx *ctx, cudaStream_t st, const float *d_vals, size_t tile_elems, uint32_t nt, unsigned *d_mm_ord, const unsigned *d_perm = nullptr);
int twi_coarse_work(tw_ctx *ctx, const float *d_coarse, unsigned cells, uint32_t nt, float level, unsigned *d_work);
int twi_gather_origins(tw_ctx *ctx, const void *d_org, const unsigned *d_order, uint32_t nt, void *d_out);
int twi_order_by_work(tw_ctx *ctx, cudaStream_t st, const unsigned *d_work, uint32_t nt, unsigned max_work, unsigned *d_hist256, unsigned *d_order);
int twi_init_minmax(tw_ctx *ctx, unsigned *d_mm_ord, uint32_t n);
