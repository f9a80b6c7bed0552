// rgs_api.cu -- the C ABI (include/rgs_b200.h): buffer carving, orchestration, error handling.
//
// Replaces CudaRasterizer::Rasterizer::{forward,backward,markVisible} and the GeometryState /
// BinningState / ImageState chunk allocator (reference: cuda_rasterizer/rasterizer_impl.cu:190-250,
// 254-425, 429-571, 176-188; cuda_rasterizer/rasterizer_impl.h:22-94).
#include <atomic>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "rgs_common.cuh"

namespace rgs {

static std::atomic<int64_t> g_launches{0};
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

static thread_local std::string t_error;

// ---- optional per-stage device timing (bench.py's roofline leg): cudaEvents recorded on the launching stream
// around each stage, read back by rgs_stage_times() after a synchronize.  Off by default: zero overhead.
enum Stage { ST_PREPROCESS, ST_SCAN, ST_BINNING, ST_RENDER_FWD, ST_RENDER_BWD, ST_PREPROCESS_BWD, ST_EXCHANGE, ST_COUNT };
static const char* kStageNames[ST_COUNT] = {"preprocess_forward", "scan", "binning_sort", "render_forward", "render_backward", "preprocess_backward", "gradient_exchange"};
struct StageRec { int stage; cudaEvent_t a, b; };
static std::mutex g_stage_mu;
static std::vector<StageRec> g_stage_pending;
static double g_stage_ms[ST_COUNT];
static int64_t g_stage_n[ST_COUNT];
static std::atomic<int> g_stage_on{0};

struct StageScope {
	cudaStream_t s; int stage; cudaEvent_t a = nullptr, b = nullptr; bool on;
	StageScope(int st, cudaStream_t stream) : s(stream), stage(st), on(g_stage_on.load() != 0) {
		if (on) { cudaEventCreate(&a); cudaEventCreate(&b); cudaEventRecord(a, s); }
	}
	~StageScope() {
		if (on) { cudaEventRecord(b, s); std::lock_guard<std::mutex> lk(g_stage_mu); g_stage_pending.push_back({stage, a, b}); }
	}
};
static void stage_collect() {
	std::lock_guard<std::mutex> lk(g_stage_mu);
	for (auto& r : g_stage_pending) {
		cudaEventSynchronize(r.b);
		float ms = 0.f;
		if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) { g_stage_ms[r.stage] += ms; g_stage_n[r.stage]++; }
		cudaEventDestroy(r.a); cudaEventDestroy(r.b);
	}
	g_stage_pending.clear();
}

static int fail(int code, const std::string& msg) {
	t_error = msg;
	return code;
}

#define RGS_CUDA_TRY(expr)                                                                                   \
	do {                                                                                                     \
		cudaError_t _e = (expr);                                                                             \
		if (_e != cudaSuccess) return fail(RGS_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
	} while (0)

// After each stage in debug mode: synchronise and surface the error, like CHECK_CUDA (auxiliary.h:404-411).
static int debug_sync(const rgs_camera* cam, cudaStream_t s, const char* stage) {
	cudaError_t e = cudaGetLastError();
	if (e == cudaSuccess && cam->debug) e = cudaStreamSynchronize(s);
	if (e != cudaSuccess) return fail(RGS_E_CUDA, std::string("[CUDA ERROR] in ") + stage + ": " + cudaGetErrorString(e));
	return RGS_OK;
}

static GeomView carve_geom(char* base, int P, bool coord, size_t* total) {
	Carver c(base);
	GeomView g;
	g.records = c.take<float>((size_t)P * rec_floats(coord));
	g.depths = c.take<float>(P);
	g.tiles_touched = c.take<uint32_t>(P);
	g.bwd_rows = c.take<uint32_t>(P);
	g.clamped = c.take<uint8_t>(P);
	g.sigma_inv = c.take<float>((size_t)P * SIGMA_INV_FLOATS);
	g.bwd_row_count = c.take<uint32_t>(1);
	if (total) *total = c.size();
	return g;
}

static BinView carve_bin(char* base, size_t R, int tiles, size_t* total) {
	Carver c(base);
	BinView b;
	b.point_list = c.take<uint32_t>(R);
	b.keys_sorted = c.take<uint64_t>(R);
	b.hitmask = c.take<uint32_t>(hitmask_words(R, tiles));
	b.keys_unsorted = c.take<uint64_t>(R);
	if (total) *total = c.size();
	return b;
}

static ImgView carve_img(char* base, int grid_x, int grid_y, size_t N, bool coord, bool depth, size_t* total) {
	const int tiles = grid_x * grid_y;
	Carver c(base);
	ImgView v;
	v.ranges = c.take<uint2>(tiles);
	v.tile_count = c.take<uint32_t>(tiles);
	v.totals = c.take<uint32_t>(2);
	v.chunk_base = c.take<uint32_t>(tiles);
	v.n_contrib = c.take<uint32_t>(2 * N);
	v.accum_depth = c.take<float>(depth ? N : 0);
	v.normal_length = c.take<float>((coord || depth) ? N : 0);
	v.accum_coord = c.take<float>(coord ? 3 * N : 0);
	v.tile_diff = c.take<int>((size_t)(grid_x + 1) * (grid_y + 1));
	if (total) *total = c.size();
	return v;
}

// Height of the [C,Hs,W] maps one call stores: the whole image, or with compact_slab only the pixel rows of tile rows
// [row_begin, row_end).
static int stored_height(const rgs_camera* cam, int row_begin, int row_end) {
	if (!cam->compact_slab) return cam->height;
	const int hs = (row_end * TILE_Y < cam->height ? row_end * TILE_Y : cam->height) - row_begin * TILE_Y;
	return hs > 0 ? hs : 0;
}

static int make_params(const rgs_camera* cam, const rgs_gaussians* g, FwdParams& p) {
	if (!cam || !g) return fail(RGS_E_INVALID, "null camera / gaussians");
	if (cam->width <= 0 || cam->height <= 0) return fail(RGS_E_INVALID, "image size must be positive");
	if (g->P < 0) return fail(RGS_E_INVALID, "negative Gaussian count");
	if (cam->prefiltered)
		return fail(RGS_E_UNSUPPORTED,
		            "prefiltered=True is mis-wired in the reference (rasterizer_impl.cu:343-345 feeds it to the `integrate` switch) and is not supported");
	const bool has_sh = g->shs != nullptr, has_col = g->colors_precomp != nullptr;
	if (has_sh == has_col && g->P > 0) return fail(RGS_E_INVALID, "Please provide excatly one of either SHs or precomputed colors!");
	const bool has_sr = g->scales != nullptr && g->rotations != nullptr, has_cov = g->cov3D_precomp != nullptr;
	if (has_sr == has_cov && g->P > 0)
		return fail(RGS_E_INVALID, "Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!");
	if (has_sh && (cam->sh_degree < 0 || cam->sh_degree > 3 || (cam->sh_degree + 1) * (cam->sh_degree + 1) > cam->sh_coeffs))
		return fail(RGS_E_INVALID, "sh_degree does not fit the stored SH coefficients");
	if (has_sh && cam->sh_coeffs > 16)
		return fail(RGS_E_INVALID, "at most 16 SH coefficients per Gaussian (degree 3) are supported");  // the SH kernels stage rows of <= 16 x 3 floats
	p.P = g->P;
	p.D = cam->sh_degree;
	p.M = has_sh ? cam->sh_coeffs : 0;
	p.W = cam->width;
	p.H = cam->height;
	p.grid_x = (cam->width + TILE_X - 1) / TILE_X;
	p.grid_y = (cam->height + TILE_Y - 1) / TILE_Y;
	p.row_begin = cam->tile_row_begin;
	p.row_end = cam->tile_row_end < 0 ? p.grid_y : cam->tile_row_end;
	if (p.row_begin < 0 || p.row_end > p.grid_y || p.row_begin > p.row_end) return fail(RGS_E_INVALID, "tile row slab out of range");
	p.py_off = cam->compact_slab ? p.row_begin * TILE_Y : 0;
	p.Hs = stored_height(cam, p.row_begin, p.row_end);
	p.tan_fovx = cam->tan_fovx;
	p.tan_fovy = cam->tan_fovy;
	// focal lengths computed on the host in float, as the reference does (rasterizer_impl.cu:288-289)
	p.focal_y = cam->height / (2.0f * cam->tan_fovy);
	p.focal_x = cam->width / (2.0f * cam->tan_fovx);
	p.kernel_size = cam->kernel_size;
	p.scale_modifier = cam->scale_modifier;
	p.coord = cam->require_coord != 0;
	p.depth = cam->require_depth != 0;
	p.means3D = g->means3D;
	p.opacities = g->opacities;
	p.shs = g->shs;
	p.shs_rest = has_sh ? g->shs_rest : nullptr;
	if (p.shs_rest != nullptr && p.M < 2) return fail(RGS_E_INVALID, "shs_rest given but sh_coeffs < 2");
	p.colors_precomp = g->colors_precomp;
	p.scales = g->scales;
	p.rotations = g->rotations;
	p.cov3D_precomp = g->cov3D_precomp;
	p.viewmatrix = cam->viewmatrix;
	p.projmatrix = cam->projmatrix;
	p.cam_pos = cam->cam_pos;
	p.background = cam->background;
	return RGS_OK;
}

// pinned 4-byte mailbox per thread for the num_rendered read-back
static uint32_t* pinned_mailbox() {
	static thread_local uint32_t* box = nullptr;
	if (!box) {
		if (cudaHostAlloc((void**)&box, 64, cudaHostAllocDefault) != cudaSuccess) box = nullptr;
	}
	return box;
}

}  // namespace rgs

using namespace rgs;

extern "C" {

const char* rgs_last_error(void) { return t_error.c_str(); }
int32_t rgs_abi_version(void) { return RGS_ABI_VERSION; }
int64_t rgs_launch_count(void) { return g_launches.load(); }
void rgs_stage_timing(int32_t enable) {
	stage_collect();
	if (enable) { std::lock_guard<std::mutex> lk(g_stage_mu); for (int i = 0; i < ST_COUNT; i++) { g_stage_ms[i] = 0; g_stage_n[i] = 0; } }
	g_stage_on.store(enable ? 1 : 0);
}
int32_t rgs_stage_times(const char** names, double* total_ms, int64_t* launches, int32_t capacity) {
	stage_collect();
	int n = capacity < ST_COUNT ? capacity : ST_COUNT;
	for (int i = 0; i < n; i++) { names[i] = kStageNames[i]; total_ms[i] = g_stage_ms[i]; launches[i] = g_stage_n[i]; }
	return n;
}
int32_t rgs_grad_stride(int32_t require_coord, int32_t /*require_depth*/) { return grad_floats(require_coord != 0); }

// preprocess -> tile counts -> (one host sync for the instance count) -> binning / sort: everything before blending.
// Shared by rgs_forward and rgs_integrate.  Returns num_rendered or a negative status.
static int64_t forward_to_binning(const rgs_camera* cam, const FwdParams& p, int* radii, const rgs_buffers* bufs, cudaStream_t s, GeomView& g,
                                  BinView& b, ImgView& img) {
	int rc;
	const int P = p.P;
	const size_t N = (size_t)p.W * p.Hs;
	const int tiles = p.grid_x * p.grid_y;

	// image-side scratch first: needed even when there is nothing to draw (background fill)
	size_t img_bytes = 0;
	carve_img(nullptr, p.grid_x, p.grid_y, N, p.coord, p.depth, &img_bytes);
	char* img_ptr = bufs->image(bufs->image_user, img_bytes);
	if (!img_ptr) return fail(RGS_E_ALLOC, "image buffer callback returned NULL");
	img = carve_img(img_ptr, p.grid_x, p.grid_y, N, p.coord, p.depth, nullptr);

	size_t geom_bytes = 0;
	carve_geom(nullptr, P, p.coord, &geom_bytes);
	char* geom_ptr = bufs->geom(bufs->geom_user, geom_bytes);
	if (!geom_ptr) return fail(RGS_E_ALLOC, "geometry buffer callback returned NULL");
	g = carve_geom(geom_ptr, P, p.coord, nullptr);

	int64_t R = 0;
	uint32_t max_list = 0;
	if (P > 0) {
		RGS_CUDA_TRY(cudaMemsetAsync(img.tile_diff, 0, (size_t)(p.grid_x + 1) * (p.grid_y + 1) * sizeof(int), s));
		{ StageScope sc(ST_PREPROCESS, s); launch_preprocess_forward(p, g, radii, img.tile_diff, s); }
		if ((rc = debug_sync(cam, s, "preprocess")) != RGS_OK) return rc;
		{ StageScope sc(ST_SCAN, s); launch_tile_scan(p, img, s); }
		// the one host sync of the forward pass: the instance count sizes the binning buffers and is returned to the
		// caller (reference: blocking cudaMemcpy, rasterizer_impl.cu:354); the longest tile list picks the sort path
		uint32_t* box = pinned_mailbox();
		if (!box) return fail(RGS_E_CUDA, "cudaHostAlloc failed for the num_rendered mailbox");
		RGS_CUDA_TRY(cudaMemcpyAsync(box, img.totals, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
		RGS_CUDA_TRY(cudaStreamSynchronize(s));
		R = (int64_t)box[0];
		max_list = box[1];
	}
	size_t bin_bytes = 0;
	carve_bin(nullptr, (size_t)R, tiles, &bin_bytes);
	char* bin_ptr = bufs->binning(bufs->binning_user, bin_bytes);
	if (!bin_ptr) return fail(RGS_E_ALLOC, "binning buffer callback returned NULL");
	b = carve_bin(bin_ptr, (size_t)R, tiles, nullptr);
	// forward-render writes a ballot word only for the chunks a warp actually tested; backward masks every position at or
	// behind the warp's last contributor, so the unwritten words never matter -- zero them anyway (<= R bytes) so that no
	// consumer (debug views, initcheck) ever sees memory the library did not write
	if (R > 0) RGS_CUDA_TRY(cudaMemsetAsync(b.hitmask, 0, hitmask_words((size_t)R, tiles) * sizeof(uint32_t), s));

	if (P == 0) {
		RGS_CUDA_TRY(cudaMemsetAsync(img.ranges, 0, (size_t)tiles * sizeof(uint2), s));
	} else {
		// lists longer than the shared-memory sort take the multi-CTA path inside launch_tile_binning
		StageScope sc(ST_BINNING, s);
		launch_tile_binning(p, g, b, img, radii, R, max_list, s);
	}
	if ((rc = debug_sync(cam, s, "binning")) != RGS_OK) return rc;
	return R;
}

int64_t rgs_forward(const rgs_camera* cam, const rgs_gaussians* gs, const rgs_forward_out* out, const rgs_buffers* bufs, void* cuda_stream) {
	FwdParams p;
	int rc = make_params(cam, gs, p);
	if (rc != RGS_OK) return rc;
	if (!out || !bufs || !bufs->geom || !bufs->binning || !bufs->image) return fail(RGS_E_INVALID, "null outputs / buffer callbacks");
	cudaStream_t s = (cudaStream_t)cuda_stream;
	GeomView g;
	BinView b;
	ImgView img;
	const int64_t R = forward_to_binning(cam, p, out->radii, bufs, s, g, b, img);
	if (R < 0) return R;
	RenderOut ro{out->out_color, out->out_coord, out->out_mcoord, out->out_alpha, out->out_normal, out->out_depth, out->out_mdepth};
	{ StageScope sc(ST_RENDER_FWD, s); launch_render_forward(p, g, b, img, ro, s); }
	if ((rc = debug_sync(cam, s, "render")) != RGS_OK) return rc;
	return R;
}

// Replaces CudaRasterizer::Rasterizer::integrate (rasterizer.h:68-108, rasterizer_impl.cu:573-844).
int64_t rgs_integrate(const rgs_camera* cam, const rgs_gaussians* gs, const rgs_integrate_io* io, const rgs_buffers* bufs, rgs_resize_fn point_buffer,
                      void* point_buffer_user, int32_t* overflowed_pixels, void* cuda_stream) {
	if (!cam) return fail(RGS_E_INVALID, "null camera / gaussians");
	rgs_camera c = *cam;
	c.require_depth = 1;  // the integrate path always carries the ray-space planes (rasterizer_impl.cu:634-668)
	c.require_coord = 0;
	c.tile_row_begin = 0;
	c.tile_row_end = -1;
	c.compact_slab = 0;
	FwdParams p;
	int rc = make_params(&c, gs, p);
	if (rc != RGS_OK) return rc;
	if (!io || !bufs || !bufs->geom || !bufs->binning || !bufs->image || !point_buffer) return fail(RGS_E_INVALID, "null outputs / buffer callbacks");
	if (io->PN <= 0 || p.P <= 0) return fail(RGS_E_INVALID, "integrate needs at least one Gaussian and one point (the reference returns its fill values)");
	if (!io->points3D || !io->out_color || !io->out_alpha_integrated || !io->out_color_integrated || !io->out_coordinate2d || !io->out_sdf || !io->radii)
		return fail(RGS_E_INVALID, "null integrate inputs / outputs");
	cudaStream_t s = (cudaStream_t)cuda_stream;
	GeomView g;
	BinView b;
	ImgView img;
	const int64_t R = forward_to_binning(&c, p, io->radii, bufs, s, g, b, img);
	if (R < 0) return R;
	const int tiles = p.grid_x * p.grid_y;
	const size_t N = (size_t)p.W * p.H;
	const int PN = io->PN;
	IntegrateView v;
	size_t bytes = 0;
	for (int pass = 0; pass < 2; pass++) {
		char* base = nullptr;
		if (pass == 1) {
			base = point_buffer(point_buffer_user, bytes);
			if (!base) return fail(RGS_E_ALLOC, "point buffer callback returned NULL");
		}
		Carver cv(base);
		v.PN = PN;
		v.points3D = io->points3D;
		v.invray = cv.take<float>((size_t)p.P * 8);
		v.masks = cv.take<uint32_t>(integrate_mask_words(R, tiles));
		v.aux = cv.take<float4>(2 * N);
		v.overflow = cv.take<int>(1);
		v.key_in = cv.take<uint32_t>(PN);
		v.key_out = cv.take<uint32_t>(PN);
		v.pid_in = cv.take<uint32_t>(PN);
		v.pid_out = cv.take<uint32_t>(PN);
		v.pxy = cv.take<float2>(PN);
		v.pdepth = cv.take<float>(PN);
		v.sort_temp_bytes = integrate_sort_temp_bytes(PN);
		v.sort_temp = cv.take<char>(v.sort_temp_bytes);
		bytes = cv.size();
	}
	IntegrateOut out{io->out_color, io->out_alpha_integrated, io->out_color_integrated, io->out_coordinate2d, io->out_sdf};
	launch_integrate(p, g, b, img, io->radii, v, out, s);
	if ((rc = debug_sync(&c, s, "integrate")) != RGS_OK) return rc;
	if (overflowed_pixels) {
		// rare diagnostic (the reference printf's from the kernel): one more small blocking read
		int host = 0;
		RGS_CUDA_TRY(cudaMemcpyAsync(&host, v.overflow, sizeof(int), cudaMemcpyDeviceToHost, s));
		RGS_CUDA_TRY(cudaStreamSynchronize(s));
		*overflowed_pixels = host;
	}
	return R;
}

static int backward_views(const rgs_camera* cam, const rgs_gaussians* gs, const rgs_backward_in* in, FwdParams& p, GeomView& g, BinView& b, ImgView& img) {
	int rc = make_params(cam, gs, p);
	if (rc != RGS_OK) return rc;
	if (!in || !in->geom_buffer || !in->image_buffer) return fail(RGS_E_INVALID, "null backward inputs / buffers");
	const size_t N = (size_t)p.W * p.Hs;
	g = carve_geom(const_cast<char*>(in->geom_buffer), p.P, p.coord, nullptr);
	b = carve_bin(const_cast<char*>(in->binning_buffer), (size_t)in->num_rendered, p.grid_x * p.grid_y, nullptr);
	img = carve_img(const_cast<char*>(in->image_buffer), p.grid_x, p.grid_y, N, p.coord, p.depth, nullptr);
	return RGS_OK;
}

int32_t rgs_backward_render(const rgs_camera* cam, const rgs_gaussians* gs, const rgs_backward_in* in, float* grad_accum, void* cuda_stream) {
	FwdParams p;
	GeomView g;
	BinView b;
	ImgView img;
	int rc = backward_views(cam, gs, in, p, g, b, img);
	if (rc != RGS_OK) return rc;
	if (p.P == 0) return RGS_OK;
	if (!grad_accum) return fail(RGS_E_INVALID, "null gradient accumulator");
	cudaStream_t s = (cudaStream_t)cuda_stream;
	RenderGradIn gin{in->dL_dout_color, in->dL_dout_coord, in->dL_dout_mcoord, in->dL_dout_depth, in->dL_dout_mdepth,
	                 in->dL_dout_alpha, in->dL_dout_normal, in->out_alpha, in->out_normal};
	{ StageScope sc(ST_RENDER_BWD, s); launch_render_backward(p, g, b, img, gin, grad_accum, s); }
	return debug_sync(cam, s, "backward render");
}

int32_t rgs_backward_render_exchange(const rgs_camera* cam, const rgs_gaussians* gs, const rgs_backward_in* in, rgs_exchange* ex, void* cuda_stream) {
	FwdParams p;
	GeomView g;
	BinView b;
	ImgView img;
	int rc = backward_views(cam, gs, in, p, g, b, img);
	if (rc != RGS_OK) return rc;
	if (p.P == 0) return RGS_OK;
	float* acc = rgs_exchange_accumulator(ex);
	if (!acc) return fail(RGS_E_INVALID, "null exchange");
	cudaStream_t s = (cudaStream_t)cuda_stream;
	RenderGradIn gin{in->dL_dout_color, in->dL_dout_coord, in->dL_dout_mcoord, in->dL_dout_depth, in->dL_dout_mdepth,
	                 in->dL_dout_alpha, in->dL_dout_normal, in->out_alpha, in->out_normal};
	{ StageScope sc(ST_RENDER_BWD, s); launch_render_backward(p, g, b, img, gin, acc, s, /*zero_first=*/false); }
	if ((rc = debug_sync(cam, s, "backward render")) != RGS_OK) return rc;
	{
		StageScope sc(ST_EXCHANGE, s);
		rc = rgs_exchange_rows(ex, p.P, g.tiles_touched, in->radii, cuda_stream);
	}
	if (rc != RGS_OK) return fail(rc, rgs_exchange_last_error());
	return debug_sync(cam, s, "gradient exchange");
}

static int32_t backward_preprocess_impl(const rgs_camera* cam, const rgs_gaussians* gs, const rgs_backward_in* in, const float* grad_accum,
                                        const rgs_backward_out* out, void* cuda_stream, bool prefilled) {
	FwdParams p;
	GeomView g;
	BinView b;
	ImgView img;
	int rc = backward_views(cam, gs, in, p, g, b, img);
	if (rc != RGS_OK) return rc;
	if (p.P == 0) return RGS_OK;
	if (!grad_accum || !out) return fail(RGS_E_INVALID, "null gradient accumulator / outputs");
	cudaStream_t s = (cudaStream_t)cuda_stream;
	ParamGradOut po{out->dL_dmeans2D, out->dL_dcolors, out->dL_dopacity, out->dL_dmeans3D, out->dL_dcov3D, out->dL_dsh, out->dL_dscales, out->dL_drotations, out->dL_dsh_rest};
	if ((p.shs_rest != nullptr) != (po.d_sh_rest != nullptr) && po.d_sh != nullptr)
		return fail(RGS_E_INVALID, "dL_dsh_rest must be given exactly when shs_rest is");
	{ StageScope sc(ST_PREPROCESS_BWD, s); launch_preprocess_backward(p, g, in->radii, grad_accum, po, s, prefilled); }
	return debug_sync(cam, s, "backward preprocess");
}

int32_t rgs_backward_preprocess(const rgs_camera* cam, const rgs_gaussians* gs, const rgs_backward_in* in, const float* grad_accum,
                                const rgs_backward_out* out, void* cuda_stream) {
	return backward_preprocess_impl(cam, gs, in, grad_accum, out, cuda_stream, false);
}

// per-device side stream + events for work that may run underneath the main stream's kernels
struct SideStream {
	cudaStream_t stream = nullptr;
	cudaEvent_t fork = nullptr, join = nullptr;
};
static SideStream* side_stream() {
	static thread_local SideStream per_dev[64];
	int dev = 0;
	if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
	SideStream& ss = per_dev[dev & 63];
	if (!ss.stream) {
		if (cudaStreamCreateWithFlags(&ss.stream, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
		if (cudaEventCreateWithFlags(&ss.fork, cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&ss.join, cudaEventDisableTiming) != cudaSuccess)
			return nullptr;
	}
	return &ss;
}

int32_t rgs_backward(const rgs_camera* cam, const rgs_gaussians* gs, const rgs_backward_in* in, const rgs_backward_out* out,
                     rgs_resize_fn grad_scratch, void* grad_scratch_user, void* cuda_stream) {
	if (!gs || !cam) return fail(RGS_E_INVALID, "null camera / gaussians");
	if (gs->P == 0) return RGS_OK;
	if (!grad_scratch) return fail(RGS_E_INVALID, "null scratch callback");
	if (!out) return fail(RGS_E_INVALID, "null gradient accumulator / outputs");
	const size_t bytes = (size_t)gs->P * grad_floats(cam->require_coord != 0) * sizeof(float);
	float* acc = reinterpret_cast<float*>(grad_scratch(grad_scratch_user, bytes));
	if (!acc) return fail(RGS_E_ALLOC, "gradient scratch callback returned NULL");
	cudaStream_t s = (cudaStream_t)cuda_stream;
	// The zero-fill of the dense gradient tensors (pure HBM writes, ~280 MB at 1 M Gaussians) runs on a side stream underneath the
	// issue-bound backward blend; everything queued on `s` before this call is ordered before it (the tensors may be recycled memory).
	bool prefilled = false;
	SideStream* ss = !cam->debug ? side_stream() : nullptr;
	if (ss) {
		FwdParams p;
		int rc0 = make_params(cam, gs, p);
		if (rc0 != RGS_OK) return rc0;
		ParamGradOut po{out->dL_dmeans2D, out->dL_dcolors, out->dL_dopacity, out->dL_dmeans3D, out->dL_dcov3D, out->dL_dsh, out->dL_dscales, out->dL_drotations, out->dL_dsh_rest};
		if (cudaEventRecord(ss->fork, s) == cudaSuccess && cudaStreamWaitEvent(ss->stream, ss->fork, 0) == cudaSuccess) {
			launch_backward_zero_fill(p, po, ss->stream);
			prefilled = cudaEventRecord(ss->join, ss->stream) == cudaSuccess;
		}
	}
	int rc = rgs_backward_render(cam, gs, in, acc, cuda_stream);
	if (prefilled && cudaStreamWaitEvent(s, ss->join, 0) != cudaSuccess) return fail(RGS_E_CUDA, "cudaStreamWaitEvent failed");
	if (rc != RGS_OK) return rc;
	return backward_preprocess_impl(cam, gs, in, acc, out, cuda_stream, prefilled);
}

int32_t rgs_mark_visible(int32_t P, const float* means3D, const float* viewmatrix, const float* /*projmatrix*/, uint8_t* present, void* cuda_stream) {
	if (P < 0) return fail(RGS_E_INVALID, "negative Gaussian count");
	if (P == 0) return RGS_OK;
	if (!means3D || !viewmatrix || !present) return fail(RGS_E_INVALID, "null pointer");
	launch_mark_visible(P, means3D, viewmatrix, present, (cudaStream_t)cuda_stream);
	cudaError_t e = cudaGetLastError();
	if (e != cudaSuccess) return fail(RGS_E_CUDA, cudaGetErrorString(e));
	return RGS_OK;
}

int32_t rgs_activate_forward(int32_t P, const float* raw_scaling, const float* raw_opacity, const float* raw_rotation, const float* filter_3D,
                             float* scales, float* opacity, float* rotations, void* cuda_stream) {
	if (P < 0) return fail(RGS_E_INVALID, "negative Gaussian count");
	if (P == 0) return RGS_OK;
	if (!raw_scaling || !raw_opacity || !raw_rotation || !filter_3D || !scales || !opacity || !rotations) return fail(RGS_E_INVALID, "null pointer");
	launch_activate_forward(P, raw_scaling, raw_opacity, raw_rotation, filter_3D, scales, opacity, rotations, (cudaStream_t)cuda_stream);
	cudaError_t e = cudaGetLastError();
	return e == cudaSuccess ? (int32_t)RGS_OK : fail(RGS_E_CUDA, cudaGetErrorString(e));
}

int32_t rgs_activate_backward(int32_t P, const float* raw_scaling, const float* raw_opacity, const float* raw_rotation, const float* filter_3D,
                              const float* g_scales, const float* g_opacity, const float* g_rotations, float* d_raw_scaling, float* d_raw_opacity,
                              float* d_raw_rotation, void* cuda_stream) {
	if (P < 0) return fail(RGS_E_INVALID, "negative Gaussian count");
	if (P == 0) return RGS_OK;
	if (!raw_scaling || !raw_opacity || !raw_rotation || !filter_3D || !g_scales || !g_opacity || !g_rotations || !d_raw_scaling || !d_raw_opacity ||
	    !d_raw_rotation)
		return fail(RGS_E_INVALID, "null pointer");
	launch_activate_backward(P, raw_scaling, raw_opacity, raw_rotation, filter_3D, g_scales, g_opacity, g_rotations, d_raw_scaling, d_raw_opacity,
	                         d_raw_rotation, (cudaStream_t)cuda_stream);
	cudaError_t e = cudaGetLastError();
	return e == cudaSuccess ? (int32_t)RGS_OK : fail(RGS_E_CUDA, cudaGetErrorString(e));
}

int32_t rgs_densification_stats(int32_t P, const float* means2D_grad, const int32_t* radii, float* grad_accum, float* grad_accum_abs,
                                float* grad_accum_abs_max, float* denom, float* max_radii2D, void* cuda_stream) {
	if (P < 0) return fail(RGS_E_INVALID, "negative Gaussian count");
	if (P == 0) return RGS_OK;
	if (!means2D_grad || !radii || !grad_accum || !grad_accum_abs || !grad_accum_abs_max || !denom) return fail(RGS_E_INVALID, "null pointer");
	launch_densification_stats(P, means2D_grad, radii, grad_accum, grad_accum_abs, grad_accum_abs_max, denom, max_radii2D, (cudaStream_t)cuda_stream);
	cudaError_t e = cudaGetLastError();
	return e == cudaSuccess ? (int32_t)RGS_OK : fail(RGS_E_CUDA, cudaGetErrorString(e));
}

static int32_t after_launch() {
	cudaError_t e = cudaGetLastError();
	return e == cudaSuccess ? (int32_t)RGS_OK : fail(RGS_E_CUDA, cudaGetErrorString(e));
}

int32_t rgs_compute_3d_filter(int32_t P, const float* xyz, int32_t n_cams, const float* cams, float focal_length, float* filter_3D,
                              float* max_distance, void* cuda_stream) {
	if (P < 0 || n_cams < 0) return fail(RGS_E_INVALID, "negative count");
	if (P == 0) return RGS_OK;
	if (!xyz || !filter_3D || !max_distance || (n_cams > 0 && !cams)) return fail(RGS_E_INVALID, "null pointer");
	if (!(focal_length > 0.0f)) return fail(RGS_E_INVALID, "focal_length must be positive");
	launch_compute_3d_filter(P, xyz, n_cams, cams, focal_length, filter_3D, max_distance, (cudaStream_t)cuda_stream);
	return after_launch();
}

int32_t rgs_ssim_l1_forward_rows(int32_t planes, int32_t H, int32_t W, int32_t row_lo, int32_t row_hi, const float* img, const float* gt, float* dmaps,
                                 double* sums, void* cuda_stream) {
	if (planes < 0 || H <= 0 || W <= 0) return fail(RGS_E_INVALID, "image size must be positive");
	if (row_lo < 0 || row_hi > H || row_lo > row_hi) return fail(RGS_E_INVALID, "row range out of the image");
	if (!img || !gt || !sums) return fail(RGS_E_INVALID, "null pointer");
	if (planes > 65535) return fail(RGS_E_INVALID, "too many image planes");
	launch_ssim_l1_forward(planes, H, W, row_lo, row_hi, img, gt, dmaps, sums, (cudaStream_t)cuda_stream);
	return after_launch();
}

int32_t rgs_ssim_l1_backward_rows(int32_t planes, int32_t H, int32_t W, int32_t row_lo, int32_t row_hi, const float* img, const float* gt,
                                  const float* dmaps, float w_ssim, float w_l1, const float* upstream, float* d_img, void* cuda_stream) {
	if (planes < 0 || H <= 0 || W <= 0) return fail(RGS_E_INVALID, "image size must be positive");
	if (row_lo < 0 || row_hi > H || row_lo > row_hi) return fail(RGS_E_INVALID, "row range out of the image");
	if (!img || !gt || !dmaps || !d_img) return fail(RGS_E_INVALID, "null pointer");
	if (planes > 65535) return fail(RGS_E_INVALID, "too many image planes");
	launch_ssim_l1_backward(planes, H, W, row_lo, row_hi, img, gt, dmaps, w_ssim, w_l1, upstream, d_img, (cudaStream_t)cuda_stream);
	return after_launch();
}

int32_t rgs_ssim_l1_forward(int32_t planes, int32_t H, int32_t W, const float* img, const float* gt, float* dmaps, double* sums, void* cuda_stream) {
	return rgs_ssim_l1_forward_rows(planes, H, W, 0, H, img, gt, dmaps, sums, cuda_stream);
}

int32_t rgs_ssim_l1_backward(int32_t planes, int32_t H, int32_t W, const float* img, const float* gt, const float* dmaps, float w_ssim, float w_l1,
                             const float* upstream, float* d_img, void* cuda_stream) {
	return rgs_ssim_l1_backward_rows(planes, H, W, 0, H, img, gt, dmaps, w_ssim, w_l1, upstream, d_img, cuda_stream);
}

int32_t rgs_normal_consistency(int32_t H, int32_t W, int32_t from_depth, float inv_fx, float inv_fy, float cx, float cy, const float* rendered_normal,
                               const float* map_expected, const float* map_median, float w_expected, float w_median, double* loss_sum,
                               float* d_normal, float* d_expected, float* d_median, void* cuda_stream) {
	if (H <= 0 || W <= 0) return fail(RGS_E_INVALID, "image size must be positive");
	if (!rendered_normal || !map_expected || !map_median || !loss_sum || !d_normal || !d_expected || !d_median) return fail(RGS_E_INVALID, "null pointer");
	launch_normal_consistency(H, W, from_depth != 0, inv_fx, inv_fy, cx, cy, rendered_normal, map_expected, map_median, w_expected, w_median, loss_sum,
	                          d_normal, d_expected, d_median, (cudaStream_t)cuda_stream);
	return after_launch();
}

int32_t rgs_debug_get_views(const rgs_camera* cam, int32_t P, int64_t num_rendered, const char* geom_buffer, const char* binning_buffer,
                            const char* image_buffer, rgs_debug_views* views) {
	if (!cam || !views) return fail(RGS_E_INVALID, "null pointer");
	const bool coord = cam->require_coord != 0, depth = cam->require_depth != 0;
	const int grid_x = (cam->width + TILE_X - 1) / TILE_X, grid_y = (cam->height + TILE_Y - 1) / TILE_Y;
	const int row_end = cam->tile_row_end < 0 ? grid_y : cam->tile_row_end;
	const size_t N = (size_t)cam->width * stored_height(cam, cam->tile_row_begin, row_end);
	GeomView g = carve_geom(const_cast<char*>(geom_buffer), P, coord, nullptr);
	BinView b = carve_bin(const_cast<char*>(binning_buffer), (size_t)num_rendered, grid_x * grid_y, nullptr);
	ImgView img = carve_img(const_cast<char*>(image_buffer), grid_x, grid_y, N, coord, depth, nullptr);
	views->point_list = b.point_list;
	views->point_list_keys = b.keys_sorted;
	views->tile_ranges = reinterpret_cast<const uint32_t*>(img.ranges);
	views->n_contrib = img.n_contrib;
	views->tiles_touched = g.tiles_touched;
	views->records = g.records;
	views->record_floats = rec_floats(coord);
	views->depths = g.depths;
	return RGS_OK;
}

}  // extern "C"
