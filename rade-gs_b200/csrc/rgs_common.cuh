// rgs_common.cuh -- shared definitions of the B200 rasterizer kernels (sm_100a only).
//
// Layouts here are private to the library (the reference treats its three byte buffers as opaque too,
// cuda_rasterizer/rasterizer_impl.h:22-94); include/rgs_b200.h is the public surface.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/rgs_b200.h"

namespace rgs {

// ---- tiling: part of the key contract (cuda_rasterizer/config.h:15-16) ----------------------------
constexpr int TILE_X = 16;
constexpr int TILE_Y = 16;
constexpr int TILE_PIX = TILE_X * TILE_Y;

// ---- packed per-Gaussian render record (written by preprocess, gathered by the render kernels) ----
// floats: 0 mx 1 my 2 conic.x 3 conic.y | 4 conic.z 5 opacity*coef 6 ray.x 7 ray.y |
//         8 r 9 g 10 b 11 t_center | 12 nx 13 ny 14 nz 15 cam_plane[5] |
//         16 vx 17 vy 18 vz 19 cam_plane[0] | 20..23 cam_plane[1..4]
// Pairs that are multiplied by a common factor in the blend sit in even/odd slots (mx,my), (ray.x,ray.y), (r,g),
// (b,t), (nx,ny): they land in aligned register pairs and go through Blackwell's packed fp32x2 FMUL2/FFMA2.
constexpr int REC_FLOATS_BASE = 16;   // variants none / depth
constexpr int REC_FLOATS_COORD = 24;  // variants coord / coord+depth

// ---- screen-space gradient accumulator (one row per Gaussian, written by backward-render) --------
// floats: 0 dmx 1 dmy | 2 dray.x 3 dray.y | 4 5 6 dcolor 7 dt | 8 9 10 dnormal 11 dopacity | 12 dconic.x 13 dconic.y
//         14 dconic.w(=yy) 15 |dm|  ||  16..18 dview_point 19..24 dcam_plane 25..31 pad
// mean2D / plane entries are stored UNSCALED (sum of dL/ddel, sum of dL_dt*d.x, ...): the constant
// factors 0.5*W, 1/focal are applied once per Gaussian in backward-preprocess.
constexpr int GRAD_FLOATS_BASE = 16;
constexpr int GRAD_FLOATS_COORD = 32;
constexpr int SIGMA_INV_FLOATS = 12;  // 9 matrix entries, flags (bit0 well-conditioned, bit1 solver converged), 2 pad

enum GradSlot {
	G_MX = 0, G_MY = 1, G_RAYX = 2, G_RAYY = 3, G_COL = 4, G_T = 7, G_NRM = 8, G_OPA = 11, G_CONX = 12, G_CONY = 13, G_CONW = 14,
	G_MABS = 15, G_VP = 16, G_CP = 19
};

__host__ __device__ inline int rec_floats(bool coord) { return coord ? REC_FLOATS_COORD : REC_FLOATS_BASE; }
__host__ __device__ inline int grad_floats(bool coord) { return coord ? GRAD_FLOATS_COORD : GRAD_FLOATS_BASE; }

// ---- buffer carving (128-byte aligned sub-arrays out of one resizable byte buffer) ----------------
struct Carver {
	char* base;
	size_t off;
	__host__ explicit Carver(char* b) : base(b), off(0) {}
	template <typename T> __host__ T* take(size_t count) {
		off = (off + 127) & ~size_t(127);
		T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
		off += count * sizeof(T);
		return p;
	}
	__host__ size_t size() const { return ((off + 127) & ~size_t(127)) + 128; }
};

struct GeomView {
	float* records;          // [P * rec_floats]
	float* depths;           // [P]  view-space z (its bit pattern is the low half of the sort key)
	uint32_t* tiles_touched; // [P]
	uint32_t* bwd_rows;      // [P]  backward preprocess: ids of the rows that received a gradient (in no particular order)
	uint8_t* clamped;        // [P]  bit c set when colour channel c was clamped at 0
	float* sigma_inv;        // [P * 12] Sigma^-1 substitute of forward (9 floats, column-major) + flags, reused by backward
	uint32_t* bwd_row_count; // [1]  length of bwd_rows
};

struct BinView {
	uint32_t* point_list;          // [R] sorted Gaussian ids
	uint64_t* keys_sorted;         // [R]
	uint32_t* hitmask;             // [(R/32 + tiles + 1) * 8] per 32-instance chunk: one ballot word per 8x4 pixel block of the tile,
	                               // written by forward-render (which splats can reach alpha >= 1/255 in the block), read by backward
	uint64_t* keys_unsorted;       // [R]  local keys (depth bits << 32 | Gaussian index) in their tile's segment, before the sort
};

struct ImgView {
	uint2* ranges;        // [tiles]
	uint32_t* tile_count; // [tiles] instances per tile (written by tile_scan_kernel from tile_diff); counted down to 0 by the scatter
	uint32_t* totals;     // [2]     num_rendered, longest tile list
	uint32_t* chunk_base; // [tiles] first 32-instance chunk of each tile in BinView::hitmask (exclusive scan of ceil(n/32))
	uint32_t* n_contrib;  // [2 * N]
	float* accum_depth;   // [N]
	float* normal_length; // [N]
	float* accum_coord;   // [3 * N]
	int* tile_diff;       // [(grid_y+1) * (grid_x+1)] corner increments of the tile rectangles; its 2D prefix sum is tile_count
};

// ---- small column-major 3x3 algebra ---------------------------------------------------------------
// Kept column-major with the reference's operator shapes (cuda_rasterizer/forward.cu:96-113 goes through
// glm): products are written a0*b0 + a1*b1 + a2*b2 left to right so that nvcc contracts them the same
// way in both builds -- this chain decides `radii` and therefore the tile keys.
struct V3 {
	float x, y, z;
};
struct M3 {
	V3 c[3];  // columns
};

__device__ __forceinline__ V3 v3(float x, float y, float z) { return V3{x, y, z}; }
__device__ __forceinline__ V3 operator+(V3 a, V3 b) { return V3{a.x + b.x, a.y + b.y, a.z + b.z}; }
__device__ __forceinline__ V3 operator-(V3 a, V3 b) { return V3{a.x - b.x, a.y - b.y, a.z - b.z}; }
__device__ __forceinline__ V3 operator*(V3 a, float s) { return V3{a.x * s, a.y * s, a.z * s}; }
__device__ __forceinline__ V3 operator*(float s, V3 a) { return V3{s * a.x, s * a.y, s * a.z}; }
__device__ __forceinline__ V3 operator/(V3 a, float s) { return V3{a.x / s, a.y / s, a.z / s}; }
__device__ __forceinline__ float dot3(V3 a, V3 b) {
	V3 t{a.x * b.x, a.y * b.y, a.z * b.z};
	return t.x + t.y + t.z;
}
__device__ __forceinline__ float at(const M3& m, int col, int row) {
	const V3& c = m.c[col];
	return row == 0 ? c.x : (row == 1 ? c.y : c.z);
}
__device__ __forceinline__ M3 m3(float x0, float y0, float z0, float x1, float y1, float z1, float x2, float y2, float z2) {
	M3 m;
	m.c[0] = V3{x0, y0, z0};
	m.c[1] = V3{x1, y1, z1};
	m.c[2] = V3{x2, y2, z2};
	return m;
}
__device__ __forceinline__ M3 transpose(const M3& m) {
	return m3(m.c[0].x, m.c[1].x, m.c[2].x, m.c[0].y, m.c[1].y, m.c[2].y, m.c[0].z, m.c[1].z, m.c[2].z);
}
__device__ __forceinline__ V3 mulcol(const M3& a, V3 b) {  // a * (column vector b)
	return V3{a.c[0].x * b.x + a.c[1].x * b.y + a.c[2].x * b.z,
	          a.c[0].y * b.x + a.c[1].y * b.y + a.c[2].y * b.z,
	          a.c[0].z * b.x + a.c[1].z * b.y + a.c[2].z * b.z};
}
__device__ __forceinline__ M3 operator*(const M3& a, const M3& b) {
	M3 r;
	r.c[0] = mulcol(a, b.c[0]);
	r.c[1] = mulcol(a, b.c[1]);
	r.c[2] = mulcol(a, b.c[2]);
	return r;
}
__device__ __forceinline__ M3 outer(V3 col, V3 row) {
	M3 r;
	r.c[0] = col * row.x;
	r.c[1] = col * row.y;
	r.c[2] = col * row.z;
	return r;
}

// ---- point transforms (cuda_rasterizer/auxiliary.h:74-113) ----------------------------------------
__device__ __forceinline__ float3 xform4x3(const float3& p, const float* m) {
	return float3{m[0] * p.x + m[4] * p.y + m[8] * p.z + m[12],
	              m[1] * p.x + m[5] * p.y + m[9] * p.z + m[13],
	              m[2] * p.x + m[6] * p.y + m[10] * p.z + m[14]};
}
__device__ __forceinline__ float4 xform4x4(const float3& p, const float* m) {
	return float4{m[0] * p.x + m[4] * p.y + m[8] * p.z + m[12],
	              m[1] * p.x + m[5] * p.y + m[9] * p.z + m[13],
	              m[2] * p.x + m[6] * p.y + m[10] * p.z + m[14],
	              m[3] * p.x + m[7] * p.y + m[11] * p.z + m[15]};
}
__device__ __forceinline__ float3 xformvec4x3T(const float3& p, const float* m) {
	return float3{m[0] * p.x + m[1] * p.y + m[2] * p.z,
	              m[4] * p.x + m[5] * p.y + m[6] * p.z,
	              m[8] * p.x + m[9] * p.y + m[10] * p.z};
}

// NDC -> pixel, evaluated in double like the reference's unsuffixed literals (auxiliary.h:57-60).
__device__ __forceinline__ float ndc_to_pix(float v, int S) { return ((v + 1.0) * S - 1.0) * 0.5; }

// Tile rectangle of a splat (auxiliary.h:62-72): float division, truncation toward zero, clamp to grid.
__device__ __forceinline__ void tile_rect(float2 p, int max_radius, int grid_x, int grid_y, uint2& rmin, uint2& rmax) {
	rmin.x = min(grid_x, max(0, (int)((p.x - max_radius) / TILE_X)));
	rmin.y = min(grid_y, max(0, (int)((p.y - max_radius) / TILE_Y)));
	rmax.x = min(grid_x, max(0, (int)((p.x + max_radius + TILE_X - 1) / TILE_X)));
	rmax.y = min(grid_y, max(0, (int)((p.y + max_radius + TILE_Y - 1) / TILE_Y)));
}

// SH basis constants (auxiliary.h:35-52; same numbers as utils/sh_utils.py:24-44).
__device__ constexpr float kSH0 = 0.28209479177387814f;
__device__ constexpr float kSH1 = 0.4886025119029199f;
__device__ constexpr float kSH2[5] = {1.0925484305920792f, -1.0925484305920792f, 0.31539156525252005f,
                                      -1.0925484305920792f, 0.5462742152960396f};
__device__ constexpr float kSH3[7] = {-0.5900435899266435f, 2.890611442640554f, -0.4570457994644658f, 0.3731763325901154f,
                                      -0.4570457994644658f, 1.445305721320277f, -0.5900435899266435f};

// ---- host-side launch bookkeeping -----------------------------------------------------------------
void count_launch(int n = 1);

// Opt a kernel in to `bytes` of dynamic shared memory on the CURRENT device (the attribute is per device and per
// function; remembered per device so the driver call happens once, also when one process drives several GPUs).
template <typename Kernel>
inline void ensure_dynamic_smem(Kernel kernel, size_t bytes, size_t (&configured)[64]) {
	int dev = 0;
	cudaGetDevice(&dev);
	dev &= 63;
	if (bytes > configured[dev]) {
		cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
		configured[dev] = bytes;
	}
}

// kernels' host launchers (one translation unit each)
struct FwdParams {
	int P, D, M, W, H;
	int grid_x, grid_y;       // tiles in the full image
	int row_begin, row_end;   // slab of tile rows handled by this call
	int py_off, Hs;           // pixel row stored first in the [C,Hs,W] maps of this call and their height (0, H unless compact_slab)
	float tan_fovx, tan_fovy, focal_x, focal_y, kernel_size, scale_modifier;
	bool coord, depth;        // variant (normal := coord || depth, forward.cu:732-739)
	const float *means3D, *opacities, *shs, *shs_rest, *colors_precomp, *scales, *rotations, *cov3D_precomp;
	const float *viewmatrix, *projmatrix, *cam_pos, *background;
};

void launch_preprocess_forward(const FwdParams& p, GeomView g, int* radii, int* tile_diff, cudaStream_t s);
void launch_mark_visible(int P, const float* means3D, const float* viewmatrix, uint8_t* present, cudaStream_t s);

// tile-bucket binning: per-tile counts -> ranges/totals -> scatter -> per-tile shared-memory sort
constexpr int TILE_SORT_CAP = 8192;   // longest tile list the one-CTA shared-memory sort takes (2 x 64 KB ping-pong); longer lists: multi-CTA chunk sort + merge
void launch_tile_scan(const FwdParams& p, ImgView img, cudaStream_t s);
void launch_tile_binning(const FwdParams& p, GeomView g, BinView b, ImgView img, const int* radii, int64_t R, uint32_t max_list, cudaStream_t s);

struct RenderOut {
	float *color, *coord, *mcoord, *alpha, *normal, *depth, *mdepth;
};
void launch_render_forward(const FwdParams& p, GeomView g, BinView b, ImgView img, RenderOut out, cudaStream_t s);
__host__ __device__ inline size_t hitmask_words(size_t R, int tiles) { return (R / 32 + (size_t)tiles + 1) * 8; }

struct RenderGradIn {
	const float *d_color, *d_coord, *d_mcoord, *d_depth, *d_mdepth, *d_alpha, *d_normal;
	const float *out_alpha, *out_normal;
};
// zero_first = false: the accumulator is known to be all-zero already (the multi-GPU exchange keeps a persistent, self-cleaning one)
void launch_render_backward(const FwdParams& p, GeomView g, BinView b, ImgView img, RenderGradIn gin, float* grad_accum, cudaStream_t s, bool zero_first = true);

struct ParamGradOut {
	float *d_means2D, *d_colors, *d_opacity, *d_means3D, *d_cov3D, *d_sh, *d_scales, *d_rotations, *d_sh_rest;
};
// prefilled: the outputs were already zero-filled by launch_backward_zero_fill (possibly on another stream, joined by the caller)
void launch_preprocess_backward(const FwdParams& p, GeomView g, const int* radii, const float* grad_accum, ParamGradOut out, cudaStream_t s,
                                bool prefilled = false);
void launch_backward_zero_fill(const FwdParams& p, ParamGradOut out, cudaStream_t s);

// fused activations / densification statistics (rgs_activation.cu; SURVEY.md 8f row 1)
void launch_activate_forward(int P, const float* raw_scaling, const float* raw_opacity, const float* raw_rotation, const float* filter_3D, float* scales,
                             float* opacity, float* rotations, cudaStream_t s);
void launch_activate_backward(int P, const float* raw_scaling, const float* raw_opacity, const float* raw_rotation, const float* filter_3D,
                              const float* g_scales, const float* g_opacity, const float* g_rotations, float* d_raw_scaling, float* d_raw_opacity,
                              float* d_raw_rotation, cudaStream_t s);
void launch_densification_stats(int P, const float* means2D_grad, const int* radii, float* grad_accum, float* grad_accum_abs, float* grad_accum_abs_max,
                                float* denom, float* max_radii2D, cudaStream_t s);

void launch_compute_3d_filter(int P, const float* xyz, int n_cams, const float* cams, float focal_length, float* filter_3D, float* max_distance,
                              cudaStream_t s);

// opacity integration at query points (rgs_integrate.cu; SURVEY.md 8f row 3)
struct IntegrateView {
	int PN;
	const float* points3D;   // [PN,3]
	float* invray;           // [P,8]  inverse ray-space covariance (6) + well-conditioned flag + pad
	uint32_t* masks;         // contribution bit masks, integrate_mask_words(R, tiles)
	float4* aux;             // [2*H*W] per-pixel state phase B needs (median splat plane, last contributor)
	int* overflow;           // pixels that hit the contributor cap
	uint32_t *key_in, *key_out, *pid_in, *pid_out;  // [PN] pixel index per point and point ids, before / after the sort
	float2* pxy;             // [PN]
	float* pdepth;           // [PN]
	char* sort_temp;
	size_t sort_temp_bytes;
};
struct IntegrateOut {
	float *out_color, *out_alpha, *out_color_int, *out_coord, *out_sdf;
};
size_t integrate_sort_temp_bytes(int PN);
size_t integrate_mask_words(int64_t R, int tiles);
void launch_integrate(const FwdParams& p, GeomView g, BinView b, ImgView img, const int* radii, IntegrateView v, IntegrateOut out, cudaStream_t s);

// fused image-side losses (rgs_image_loss.cu; SURVEY.md 8f row 2)
void launch_ssim_l1_forward(int planes, int H, int W, int row_lo, int row_hi, const float* img, const float* gt, float* dmaps, double* sums,
                            cudaStream_t s);
void launch_ssim_l1_backward(int planes, int H, int W, int row_lo, int row_hi, const float* img, const float* gt, const float* dmaps, float w_ssim,
                             float w_l1, const float* upstream, float* d_img, cudaStream_t s);
void launch_normal_consistency(int H, int W, bool from_depth, float inv_fx, float inv_fy, float cx, float cy, const float* rendered_normal,
                               const float* map_e, const float* map_m, float w_e, float w_m, double* loss_sum, float* d_normal, float* d_e, float* d_m,
                               cudaStream_t s);

}  // namespace rgs
