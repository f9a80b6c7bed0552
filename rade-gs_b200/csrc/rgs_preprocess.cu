// rgs_preprocess.cu -- per-Gaussian forward preprocess for sm_100a.
//
// Replaces preprocessCUDA<3,false> + computeCov3D + computeCov2D<false> + computeColorFromSH
// (reference: cuda_rasterizer/forward.cu:23-74, 77-264, 270-304, 307-423) and checkFrustum
// (cuda_rasterizer/rasterizer_impl.cu:54-66).
//
// What is different from the reference (by design, results within tolerance; keys bit-exact):
//   * one packed 64/96-byte render record per Gaussian instead of nine SoA arrays;
//   * the 3x3 symmetric eigen-decomposition of Sigma keeps the reference's algorithm and absolute stopping
//     tests (rgs_geom.cuh explains why a more accurate one would break parity of the normal map);
//   * the key-determining chain (p_view.z, NDC->pixel, cov2D -> radius -> tile rect) keeps the
//     reference's expression shapes so both builds round identically.
#include <math_constants.h>

#include "rgs_geom.cuh"

namespace rgs {

// SH -> RGB (forward.cu:23-74).  `sh` points at this Gaussian's [M,3] block; with the split layout (`rest` != NULL)
// `sh` is its [1,3] coefficient-0 row and `rest` its [M-1,3] block of the higher bands.
__device__ __forceinline__ float3 sh_to_rgb(int deg, int M, const float* __restrict__ sh, const float* __restrict__ rest, float3 pos, float3 campos,
                                            uint8_t& clamp_bits) {
	float3 dir = {pos.x - campos.x, pos.y - campos.y, pos.z - campos.z};
	float len = sqrtf(dir.x * dir.x + dir.y * dir.y + dir.z * dir.z);
	dir.x /= len; dir.y /= len; dir.z /= len;

	// Coefficients are consumed band by band (3, 9, 15, 21 floats) so that at most one band is live in registers; the
	// per-channel sum keeps the reference's left-to-right order (forward.cu:39-66) and so the same FMA contraction.
	const float* hi = rest != nullptr ? rest - 3 : sh;  // coefficient k >= 1 starts at hi + 3k in both layouts
	// 128-bit loads only when every Gaussian's block is a whole number of float4 (M = 4, 8, 12, 16): no read past a block's end
	const bool vec = rest == nullptr && ((3 * M) & 3) == 0 && (reinterpret_cast<uintptr_t>(sh) & 15) == 0;
	float res[3];
	const float x = dir.x, y = dir.y, z = dir.z;
	float b[24];
	// band 0 (+ band 1: floats 0..11 are exactly three aligned float4 in the concatenated layout)
	if (vec) {
		const float4* s4 = reinterpret_cast<const float4*>(sh);
		const float4 v0 = __ldg(s4);
		b[0] = v0.x; b[1] = v0.y; b[2] = v0.z; b[3] = v0.w;
		if (deg > 0) {
			const float4 v1 = __ldg(s4 + 1), v2 = __ldg(s4 + 2);
			b[4] = v1.x; b[5] = v1.y; b[6] = v1.z; b[7] = v1.w; b[8] = v2.x; b[9] = v2.y; b[10] = v2.z; b[11] = v2.w;
		}
	} else {
		b[0] = __ldg(sh); b[1] = __ldg(sh + 1); b[2] = __ldg(sh + 2);
		if (deg > 0) {
#pragma unroll
			for (int i = 3; i < 12; i++) b[i] = __ldg(hi + i);
		}
	}
	// The basis polynomials are evaluated BEFORE each band's (layout-dependent) loads and with the reference's expression
	// trees ((k * y) * (3xx - yy)) * sh: what follows the loads is then a chain of a*b+c steps that can contract in one way
	// only, so both layouts round identically whatever the compiler does with the two load paths.
	const float B1 = kSH1 * y, B2 = kSH1 * z, B3 = kSH1 * x;
#pragma unroll
	for (int ch = 0; ch < 3; ch++) {
		float r = kSH0 * b[ch];
		if (deg > 0) r = r - B1 * b[3 + ch] + B2 * b[6 + ch] - B3 * b[9 + ch];
		res[ch] = r;
	}
	if (deg > 1) {
		const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
		const float B4 = kSH2[0] * xy, B5 = kSH2[1] * yz, B6 = kSH2[2] * (2.0f * zz - xx - yy), B7 = kSH2[3] * xz, B8 = kSH2[4] * (xx - yy);
		float B9 = 0.f, B10 = 0.f, B11 = 0.f, B12 = 0.f, B13 = 0.f, B14 = 0.f, B15 = 0.f;
		if (deg > 2) {
			B9 = kSH3[0] * y * (3.0f * xx - yy); B10 = kSH3[1] * xy * z; B11 = kSH3[2] * y * (4.0f * zz - xx - yy);
			B12 = kSH3[3] * z * (2.0f * zz - 3.0f * xx - 3.0f * yy); B13 = kSH3[4] * x * (4.0f * zz - xx - yy); B14 = kSH3[5] * z * (xx - yy);
			B15 = kSH3[6] * x * (xx - 3.0f * yy);
		}
		// band 2: floats 12..26 (coefficients 4..8); floats 12..27 are four aligned float4, the last one carries float 27
		float carry = 0.f;
		if (vec) {
			const float4* s4 = reinterpret_cast<const float4*>(sh) + 3;
#pragma unroll
			for (int i = 0; i < 4; i++) {
				const float4 v = __ldg(s4 + i);
				b[4 * i] = v.x; b[4 * i + 1] = v.y; b[4 * i + 2] = v.z; b[4 * i + 3] = v.w;
			}
			carry = b[15];
		} else {
#pragma unroll
			for (int i = 0; i < 15; i++) b[i] = __ldg(hi + 12 + i);
		}
#pragma unroll
		for (int ch = 0; ch < 3; ch++) res[ch] = res[ch] + B4 * b[ch] + B5 * b[3 + ch] + B6 * b[6 + ch] + B7 * b[9 + ch] + B8 * b[12 + ch];
		if (deg > 2) {
			// band 3: floats 27..47 (coefficients 9..15)
			if (vec) {
				const float4* s4 = reinterpret_cast<const float4*>(sh) + 7;
				b[0] = carry;
#pragma unroll
				for (int i = 0; i < 5; i++) {
					const float4 v = __ldg(s4 + i);
					b[1 + 4 * i] = v.x; b[2 + 4 * i] = v.y; b[3 + 4 * i] = v.z; b[4 + 4 * i] = v.w;
				}
			} else {
#pragma unroll
				for (int i = 0; i < 21; i++) b[i] = __ldg(hi + 27 + i);
			}
#pragma unroll
			for (int ch = 0; ch < 3; ch++)
				res[ch] = res[ch] + B9 * b[ch] + B10 * b[3 + ch] + B11 * b[6 + ch] + B12 * b[9 + ch] + B13 * b[12 + ch] + B14 * b[15 + ch] +
				          B15 * b[18 + ch];
		}
	}
#pragma unroll
	for (int ch = 0; ch < 3; ch++) res[ch] += 0.5f;
	clamp_bits = (res[0] < 0 ? 1 : 0) | (res[1] < 0 ? 2 : 0) | (res[2] < 0 ? 4 : 0);
	return float3{fmaxf(res[0], 0.0f), fmaxf(res[1], 0.0f), fmaxf(res[2], 0.0f)};
}

// 64 registers, 4 CTAs per SM: 5-10 % faster than 3 CTAs per SM on C2 / C3
__global__ void __launch_bounds__(256, 4) preprocess_forward_kernel(FwdParams p, GeomView g, int* __restrict__ radii, int* __restrict__ tile_diff) {
	const int idx = blockIdx.x * blockDim.x + threadIdx.x;
	if (idx >= p.P) return;

	// Not rendered unless proven otherwise (forward.cu:346-349).
	int my_radii = 0;
	uint32_t my_tiles = 0;

	const float* V = p.viewmatrix;
	const float3 p_orig = {p.means3D[3 * idx], p.means3D[3 * idx + 1], p.means3D[3 * idx + 2]};
	const float3 p_view = xform4x3(p_orig, V);

	// near-plane cull only (auxiliary.h:170)
	if (p_view.z > 0.2f) {
		const float4 p_hom = xform4x4(p_orig, p.projmatrix);
		const float p_w = 1.0f / (p_hom.w + 0.0000001f);
		const float3 p_proj = {p_hom.x * p_w, p_hom.y * p_w, p_hom.z * p_w};

		// ---- 3D covariance (forward.cu:270-304) ----
		float cov3D[6];
		if (p.cov3D_precomp != nullptr) {
#pragma unroll
			for (int i = 0; i < 6; i++) cov3D[i] = p.cov3D_precomp[6 * idx + i];
		} else {
			const float sx = p.scales[3 * idx], sy = p.scales[3 * idx + 1], sz = p.scales[3 * idx + 2];
			const float4 q = *reinterpret_cast<const float4*>(p.rotations + 4 * idx);
			M3 S = m3(p.scale_modifier * sx, 0.f, 0.f, 0.f, p.scale_modifier * sy, 0.f, 0.f, 0.f, p.scale_modifier * sz);
			const M3 Rg = quat_to_glm_rot(q.x, q.y, q.z, q.w);
			M3 Mm = S * Rg;
			M3 Sigma = transpose(Mm) * Mm;
			cov3D[0] = Sigma.c[0].x; cov3D[1] = Sigma.c[0].y; cov3D[2] = Sigma.c[0].z;
			cov3D[3] = Sigma.c[1].y; cov3D[4] = Sigma.c[1].z; cov3D[5] = Sigma.c[2].z;
		}

		// ---- EWA 2D covariance (forward.cu:85-124); this chain decides the radius ----
		float3 t = p_view;
		const float limx = 1.3f * p.tan_fovx;
		const float limy = 1.3f * p.tan_fovy;
		float txtz = t.x / t.z;
		float tytz = t.y / t.z;
		t.x = min(limx, max(-limx, txtz)) * t.z;
		t.y = min(limy, max(-limy, tytz)) * t.z;
		txtz = t.x / t.z;
		tytz = t.y / t.z;

		M3 J = m3(p.focal_x / t.z, 0.0f, -(p.focal_x * t.x) / (t.z * t.z),
		          0.0f, p.focal_y / t.z, -(p.focal_y * t.y) / (t.z * t.z),
		          0.f, 0.f, 0.f);
		M3 Wm = m3(V[0], V[4], V[8], V[1], V[5], V[9], V[2], V[6], V[10]);
		M3 T = Wm * J;
		M3 Vrk = m3(cov3D[0], cov3D[1], cov3D[2], cov3D[1], cov3D[3], cov3D[4], cov3D[2], cov3D[4], cov3D[5]);
		M3 cov = transpose(T) * transpose(Vrk) * T;

		const float c00 = cov.c[0].x, c01 = cov.c[0].y, c11 = cov.c[1].y;
		const float3 cov2 = {float(c00 + p.kernel_size), float(c01), float(c11 + p.kernel_size)};
		const float det_0 = max(1e-6, c00 * c11 - c01 * c01);
		const float det_1 = max(1e-6, (c00 + p.kernel_size) * (c11 + p.kernel_size) - c01 * c01);
		float coef = sqrt(det_0 / (det_1 + 1e-6) + 1e-6);
		if (det_0 <= 1e-6 || det_1 <= 1e-6) coef = 0.0f;

		// Invert covariance (forward.cu:385-389)
		const float det = (cov2.x * cov2.z - cov2.y * cov2.y);
		if (det != 0.0f) {
			const float det_inv = 1.f / det;
			const float3 conic = {cov2.z * det_inv, -cov2.y * det_inv, cov2.x * det_inv};

			// extent -> tile rectangle (forward.cu:395-403)
			const float mid = 0.5f * (cov2.x + cov2.z);
			const float lambda1 = mid + sqrt(max(0.1f, mid * mid - det));
			const float lambda2 = mid - sqrt(max(0.1f, mid * mid - det));
			const float my_radius = ceil(3.f * sqrt(max(lambda1, lambda2)));
			const float2 point_image = {ndc_to_pix(p_proj.x, p.W), ndc_to_pix(p_proj.y, p.H)};
			uint2 rect_min, rect_max;
			tile_rect(point_image, my_radius, p.grid_x, p.grid_y, rect_min, rect_max);
			if ((rect_max.x - rect_min.x) * (rect_max.y - rect_min.y) != 0) {
				// ---- geometry terms: ray-space plane, camera-space plane, normal (forward.cu:135-262) ----
				float cam_plane[6] = {0, 0, 0, 0, 0, 0};
				float2 ray_plane = {0.f, 0.f};
				float3 normal = {0.f, 0.f, 0.f};
				if (p.coord || p.depth) {
					const SigmaInv si = sigma_inverse(cov3D);
					{
						// keep Sigma^-1 for backward-preprocess: it would otherwise repeat the (divergent) eigen-solver
						float4* sv = reinterpret_cast<float4*>(g.sigma_inv + (size_t)idx * SIGMA_INV_FLOATS);
						sv[0] = make_float4(si.inv.c[0].x, si.inv.c[0].y, si.inv.c[0].z, si.inv.c[1].x);
						sv[1] = make_float4(si.inv.c[1].y, si.inv.c[1].z, si.inv.c[2].x, si.inv.c[2].y);
						sv[2] = make_float4(si.inv.c[2].z, __int_as_float((si.well ? 1 : 0) | (si.solved ? 2 : 0)), 0.f, 0.f);
					}
					const M3 cov_cam_inv = transpose(Wm) * si.inv * Wm;
					const V3 uvh = {txtz, tytz, 1.f};
					const V3 uvh_m = mulcol(cov_cam_inv, uvh);
					const V3 uvh_mn = uvh_m * (1.0f / sqrtf(dot3(uvh_m, uvh_m)));
					if (!isnan(uvh_mn.x) && si.solved) {
						const float u2 = txtz * txtz, v2 = tytz * tytz, uv = txtz * tytz;
						const float l = sqrt(t.x * t.x + t.y * t.y + t.z * t.z);
						const float vbn = dot3(uvh_mn, uvh);
						const float nl = u2 + v2 + 1;
						const float factor_normal = l / nl;
						const V3 q = uvh_mn / max(vbn, 0.0000001f);
						const float plane0 = (v2 + 1) * q.x + (-uv) * q.y + (-txtz) * q.z;
						const float plane1 = (-uv) * q.x + (u2 + 1) * q.y + (-tytz) * q.z;
						cam_plane[0] = (-(v2 + 1) * t.z + plane0 * t.x) / nl / p.focal_x;
						cam_plane[1] = (uv * t.z + plane1 * t.x) / nl / p.focal_y;
						cam_plane[2] = (uv * t.z + plane0 * t.y) / nl / p.focal_x;
						cam_plane[3] = (-(u2 + 1) * t.z + plane1 * t.y) / nl / p.focal_y;
						cam_plane[4] = (t.x + plane0 * t.z) / nl / p.focal_x;
						cam_plane[5] = (t.y + plane1 * t.z) / nl / p.focal_y;
						ray_plane = {plane0 * l / nl / p.focal_x, plane1 * l / nl / p.focal_y};
						const V3 rn = {-plane0 * factor_normal, -plane1 * factor_normal, -1.f};
						// nJ * rn with nJ columns (1/tz, 0, -tx/tz^2), (0, 1/tz, -ty/tz^2), (tx/l, ty/l, tz/l)  (forward.cu:176-179,257)
						const M3 nJ = m3(1 / t.z, 0.0f, -(t.x) / (t.z * t.z), 0.0f, 1 / t.z, -(t.y) / (t.z * t.z), t.x / l, t.y / l, t.z / l);
						const V3 cn = mulcol(nJ, rn);
						const float cinv = 1.0f / sqrtf(dot3(cn, cn));
						normal = {cn.x * cinv, cn.y * cinv, cn.z * cinv};
					}
				}

				// ---- colour (forward.cu:405-413) ----
				float3 rgb;
				uint8_t clamp_bits = 0;
				if (p.colors_precomp == nullptr) {
					const float3 campos = {p.cam_pos[0], p.cam_pos[1], p.cam_pos[2]};
					if (p.shs_rest != nullptr)
						rgb = sh_to_rgb(p.D, p.M, p.shs + (size_t)idx * 3, p.shs_rest + (size_t)idx * (p.M - 1) * 3, p_orig, campos, clamp_bits);
					else
						rgb = sh_to_rgb(p.D, p.M, p.shs + (size_t)idx * p.M * 3, nullptr, p_orig, campos, clamp_bits);
				} else {
					rgb = {p.colors_precomp[3 * idx], p.colors_precomp[3 * idx + 1], p.colors_precomp[3 * idx + 2]};
				}
				g.clamped[idx] = clamp_bits;

				const float ts = sqrt(p_view.x * p_view.x + p_view.y * p_view.y + p_view.z * p_view.z);
				const float opac = p.opacities[idx] * coef;

				// ---- packed record ----
				const int RF = rec_floats(p.coord);
				float4* rec = reinterpret_cast<float4*>(g.records + (size_t)idx * RF);
				rec[0] = make_float4(point_image.x, point_image.y, conic.x, conic.y);
				rec[1] = make_float4(conic.z, opac, ray_plane.x, ray_plane.y);
				rec[2] = make_float4(rgb.x, rgb.y, rgb.z, ts);
				rec[3] = make_float4(normal.x, normal.y, normal.z, cam_plane[5]);
				if (p.coord) {
					rec[4] = make_float4(p_view.x, p_view.y, p_view.z, cam_plane[0]);
					rec[5] = make_float4(cam_plane[1], cam_plane[2], cam_plane[3], cam_plane[4]);
				}
				g.depths[idx] = p_view.z;
				my_radii = (int)my_radius;
				// tiles of THIS call's slab of tile rows (whole image on a single GPU)
				const int ry0 = max((int)rect_min.y, p.row_begin);
				const int ry1 = min((int)rect_max.y, p.row_end);
				my_tiles = (rect_max.x - rect_min.x) * (uint32_t)max(0, ry1 - ry0);
				// tile-bucket binning needs the instances per tile.  Instead of one increment per covered tile (9 on average,
				// unbounded for large splats) the rectangle leaves +1 / -1 at its four corners of a (grid_y+1) x (grid_x+1)
				// difference grid; the 2D prefix sum taken by tile_scan_kernel turns that into the exact per-tile counts.
				if (tile_diff != nullptr && my_tiles != 0) {
					const int W1 = p.grid_x + 1, xa = (int)rect_min.x, xb = (int)rect_max.x;
					atomicAdd(tile_diff + ry0 * W1 + xa, 1);
					atomicAdd(tile_diff + ry0 * W1 + xb, -1);
					atomicAdd(tile_diff + ry1 * W1 + xa, -1);
					atomicAdd(tile_diff + ry1 * W1 + xb, 1);
				}
			}
		}
	}
	radii[idx] = my_radii;
	g.tiles_touched[idx] = my_tiles;
}

void launch_preprocess_forward(const FwdParams& p, GeomView g, int* radii, int* tile_diff, cudaStream_t s) {
	const int threads = 256;
	const int blocks = (p.P + threads - 1) / threads;
	preprocess_forward_kernel<<<blocks, threads, 0, s>>>(p, g, radii, tile_diff);
	count_launch();
}

__global__ void mark_visible_kernel(int P, const float* __restrict__ means3D, const float* __restrict__ V, uint8_t* __restrict__ present) {
	const int idx = blockIdx.x * blockDim.x + threadIdx.x;
	if (idx >= P) return;
	const float3 p_orig = {means3D[3 * idx], means3D[3 * idx + 1], means3D[3 * idx + 2]};
	const float3 p_view = xform4x3(p_orig, V);
	present[idx] = p_view.z > 0.2f ? 1 : 0;
}

void launch_mark_visible(int P, const float* means3D, const float* viewmatrix, uint8_t* present, cudaStream_t s) {
	mark_visible_kernel<<<(P + 255) / 256, 256, 0, s>>>(P, means3D, viewmatrix, present);
	count_launch();
}

}  // namespace rgs
