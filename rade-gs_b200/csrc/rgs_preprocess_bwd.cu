// rgs_preprocess_bwd.cu -- per-Gaussian backward preprocess for sm_100a.
//
// Replaces, fused into one kernel, computeCov2DCUDA + preprocessCUDA<3> backward with
// computeColorFromSH / computeCov3D backward (reference: cuda_rasterizer/backward.cu:145-488, 560-628,
// 21-140, 492-555).  Input is the packed screen-space gradient row written by backward-render; output
// is every parameter gradient the API returns, fully written (zeros for Gaussians that were not rendered),
// so the host allocates with empty() instead of fourteen zero-fills (rasterize_points.cu:180-193).
//
// Faithfulness notes (SURVEY.md appendix A):
//   * the hand-derived, epsilon-regularised gradient of the mip coefficient is restated as is, INCLUDING the
//     reference's aliasing bug: BACKWARD::preprocess receives dL_dconic where conic_opacity is expected
//     (rasterizer_impl.cu:569 vs backward.h:94), so `combined_opacity` below is dL_dconic.w.  Set
//     RGS_FIX_MIP_GRADIENT to use the true opacity*coef instead (off by default: parity first);
//   * gradients are w.r.t. the quaternion as given (no normalisation inside, backward.cu:554);
//   * Sigma's eigen-decomposition follows the reference's solver and stopping rules (see rgs_geom.cuh).
#include <cstdlib>

#include "rgs_geom.cuh"

namespace rgs {

// One Gaussian's parameter gradients from its accumulator row.  Writes every output of the row (zeros when not rendered / nothing received).
__device__ __forceinline__ void preprocess_backward_row(const FwdParams& p, const GeomView& g, const int* __restrict__ radii,
                                                        const float* __restrict__ grad_accum, const ParamGradOut& out, int fix_mip, const int idx) {
	bool visible = radii[idx] > 0;

	float o_means2D[3] = {0, 0, 0}, o_colors[3] = {0, 0, 0}, o_opacity = 0.f, o_mean3D[3] = {0, 0, 0};
	float o_cov[6] = {0, 0, 0, 0, 0, 0}, o_scale[3] = {0, 0, 0}, o_rot[4] = {0, 0, 0, 0};

	float gr[GRAD_FLOATS_COORD];
	if (visible) {
		const int GF = grad_floats(p.coord);
		const float* ga = grad_accum + (size_t)idx * GF;
		bool any = false;
#pragma unroll
		for (int i = 0; i < GRAD_FLOATS_BASE / 4; i++) {
			const float4 v = *reinterpret_cast<const float4*>(ga + 4 * i);
			gr[4 * i] = v.x; gr[4 * i + 1] = v.y; gr[4 * i + 2] = v.z; gr[4 * i + 3] = v.w;
			any = any || v.x != 0.f || v.y != 0.f || v.z != 0.f || v.w != 0.f;
		}
		if (p.coord) {
#pragma unroll
			for (int i = GRAD_FLOATS_BASE / 4; i < GRAD_FLOATS_COORD / 4; i++) {
				const float4 v = *reinterpret_cast<const float4*>(ga + 4 * i);
				gr[4 * i] = v.x; gr[4 * i + 1] = v.y; gr[4 * i + 2] = v.z; gr[4 * i + 3] = v.w;
				any = any || v.x != 0.f || v.y != 0.f || v.z != 0.f || v.w != 0.f;
			}
		} else {
#pragma unroll
			for (int i = GRAD_FLOATS_BASE; i < GRAD_FLOATS_COORD; i++) gr[i] = 0.f;
		}
		// A rendered splat no pixel received (occluded, or below 1/255 everywhere) has an all-zero row: every output of the chain
		// below is a sum of products with those zeros (the reference computes exactly 0 for it), so skip the chain and its loads.
		// NaN rows compare unequal to zero and take the full path.
		visible = any;
	}
	if (visible) {

		const float* V = p.viewmatrix;
		const float h_x = p.focal_x, h_y = p.focal_y;
		const float ddelx_dx = 0.5 * p.W, ddely_dy = 0.5 * p.H;

		// ---- gradients handed over by backward-render, constant factors applied here ----
		const float3 dL_dconic = {gr[G_CONX], gr[G_CONY], gr[G_CONW]};
		const V3 dL_dnormal = {gr[G_NRM], gr[G_NRM + 1], gr[G_NRM + 2]};
		const float2 dcp0 = {gr[G_CP + 0] / h_x, gr[G_CP + 1] / h_y};
		const float2 dcp1 = {gr[G_CP + 2] / h_x, gr[G_CP + 3] / h_y};
		const float2 dcp2 = {gr[G_CP + 4] / h_x, gr[G_CP + 5] / h_y};
		const float2 dray = {gr[G_RAYX] / h_x, gr[G_RAYY] / h_y};
		const float dL_dts = gr[G_T];
		const float3 dL_dview_point = {gr[G_VP], gr[G_VP + 1], gr[G_VP + 2]};
		const float2 dL_dmean2D = {gr[G_MX] * ddelx_dx, gr[G_MY] * ddely_dy};
		float dL_dopacity = gr[G_OPA];
		o_means2D[0] = dL_dmean2D.x; o_means2D[1] = dL_dmean2D.y; o_means2D[2] = gr[G_MABS];
		o_colors[0] = gr[G_COL]; o_colors[1] = gr[G_COL + 1]; o_colors[2] = gr[G_COL + 2];

		// ---- recompute forward intermediates (backward.cu:166-252) ----
		const float3 mean = {p.means3D[3 * idx], p.means3D[3 * idx + 1], p.means3D[3 * idx + 2]};
		float cov3D[6];
		M3 Rg = m3(1, 0, 0, 0, 1, 0, 0, 0, 1);
		V3 s_mod = {0, 0, 0};
		float4 q = {1, 0, 0, 0};
		const bool from_scales = (p.cov3D_precomp == nullptr);
		if (!from_scales) {
#pragma unroll
			for (int i = 0; i < 6; i++) cov3D[i] = p.cov3D_precomp[6 * idx + i];
		} else {
			q = *reinterpret_cast<const float4*>(p.rotations + 4 * idx);
			s_mod = V3{p.scale_modifier * p.scales[3 * idx], p.scale_modifier * p.scales[3 * idx + 1], p.scale_modifier * p.scales[3 * idx + 2]};
			M3 S = m3(s_mod.x, 0.f, 0.f, 0.f, s_mod.y, 0.f, 0.f, 0.f, s_mod.z);
			Rg = quat_to_glm_rot(q.x, q.y, q.z, q.w);
			M3 Mm = S * Rg;
			M3 Sigma = transpose(Mm) * Mm;
			cov3D[0] = Sigma.c[0].x; cov3D[1] = Sigma.c[0].y; cov3D[2] = Sigma.c[0].z;
			cov3D[3] = Sigma.c[1].y; cov3D[4] = Sigma.c[1].z; cov3D[5] = Sigma.c[2].z;
		}

		float3 t = xform4x3(mean, V);
		const float limx = 1.3f * p.tan_fovx, limy = 1.3f * p.tan_fovy;
		float txtz = t.x / t.z, tytz = t.y / t.z;
		t.x = min(limx, max(-limx, txtz)) * t.z;
		t.y = min(limy, max(-limy, tytz)) * t.z;
		const float x_grad_mul = txtz < -limx || txtz > limx ? 0 : 1;
		const float y_grad_mul = tytz < -limy || tytz > limy ? 0 : 1;
		txtz = t.x / t.z;
		tytz = t.y / t.z;

		M3 J = m3(h_x / t.z, 0.0f, -(h_x * t.x) / (t.z * t.z), 0.0f, h_y / t.z, -(h_y * t.y) / (t.z * t.z), 0.f, 0.f, 0.f);
		M3 Wm = m3(V[0], V[4], V[8], V[1], V[5], V[9], V[2], V[6], V[10]);
		M3 Vrk = m3(cov3D[0], cov3D[1], cov3D[2], cov3D[1], cov3D[3], cov3D[4], cov3D[2], cov3D[4], cov3D[5]);
		M3 T = Wm * J;
		M3 cov2D = transpose(T) * transpose(Vrk) * T;
		const float c00 = cov2D.c[0].x, c01 = cov2D.c[0].y, c11 = cov2D.c[1].y;
		const float ks = p.kernel_size;
		const float det_0 = max(1e-6, c00 * c11 - c01 * c01);
		const float det_1 = max(1e-6, (c00 + ks) * (c11 + ks) - c01 * c01);
		const float coef = sqrt(det_0 / (det_1 + 1e-6) + 1e-6);

		// ---- geometry backward: planes / normal -> Sigma, t (backward.cu:221-365) ----
		const float u2 = txtz * txtz, v2 = tytz * tytz, uv = txtz * tytz;
		float dVrk[6] = {0, 0, 0, 0, 0, 0};  // symmetric-summed: xx, xy+yx, xz+zx, yy, yz+zy, zz
		float plane0 = 0.f, plane1 = 0.f, dL_du = 0.f, dL_dv = 0.f, dL_dl = 0.f, l = 1.f, nl = 1.f;
		V3 dcn = {0, 0, 0}, rn = {0, 0, 0};  // dL_dnJ = dcn * rn^T
		if (p.coord || p.depth) {
			// Sigma^-1 as forward computed it (bit-identical, stored in the geometry buffer); only the rare rank-1 branch
			// needs the eigenvectors again and re-runs the solver
			SigmaInv si;
			{
				const float4* sv = reinterpret_cast<const float4*>(g.sigma_inv + (size_t)idx * SIGMA_INV_FLOATS);
				const float4 s0 = sv[0], s1 = sv[1], s2 = sv[2];
				si.inv = m3(s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w, s2.x);
				const int fl = __float_as_int(s2.y);
				si.well = (fl & 1) != 0;
				si.solved = (fl & 2) != 0;
				si.min_id = 0;
				si.lam_min = 0.f;
				if (!si.well) si = sigma_inverse(cov3D);
			}
			const M3& Vrk_inv = si.inv;
			const M3 cov_cam_inv = transpose(Wm) * Vrk_inv * Wm;
			const V3 uvh = {txtz, tytz, 1.f};
			const V3 uvh_m = mulcol(cov_cam_inv, uvh);
			const V3 uvh_mn = uvh_m * (1.0f / sqrtf(dot3(uvh_m, uvh_m)));
			if (!isnan(uvh_mn.x) && si.solved) {
				const float vb = dot3(uvh_m, uvh);
				const float vbn = dot3(uvh_mn, uvh);
				l = sqrt(t.x * t.x + t.y * t.y + t.z * t.z);
				const M3 nJ = m3(1 / t.z, 0.0f, -(t.x) / (t.z * t.z), 0.0f, 1 / t.z, -(t.y) / (t.z * t.z), t.x / l, t.y / l, t.z / l);
				const M3 nJ_inv = m3(v2 + 1, -uv, 0.f, -uv, u2 + 1, 0.f, -txtz, -tytz, 0.f);
				const float clamp_vb = max(vb, 0.0000001f);
				const float clamp_vbn = max(vbn, 0.0000001f);
				nl = u2 + v2 + 1;
				const float factor_normal = l / nl;
				const V3 qv = uvh_mn / clamp_vbn;  // uvh_m_vb
				const V3 plane = mulcol(nJ_inv, qv);
				plane0 = plane.x;
				plane1 = plane.y;
				const float2 cp0 = {(-(v2 + 1) * t.z + plane0 * t.x) / nl, (uv * t.z + plane1 * t.x) / nl};
				const float2 cp1 = {(uv * t.z + plane0 * t.y) / nl, (-(u2 + 1) * t.z + plane1 * t.y) / nl};
				const float2 cp2 = {(t.x + plane0 * t.z) / nl, (t.y + plane1 * t.z) / nl};
				const float2 ray_plane = {plane0 * factor_normal, plane1 * factor_normal};
				rn = V3{-plane0 * factor_normal, -plane1 * factor_normal, -1.f};
				const V3 cn = mulcol(nJ, rn);
				const V3 nvec = cn * (1.0f / sqrtf(dot3(cn, cn)));
				const float lv = sqrtf(dot3(cn, cn));
				const V3 dn_lv = dL_dnormal / lv;
				dcn = dn_lv - nvec * dot3(nvec, dn_lv);
				const V3 drn = mulcol(transpose(nJ), dcn);
				dL_dl = (-plane0 * drn.x - plane1 * drn.y + plane0 * dray.x + plane1 * dray.y) / nl;
				const float dpx = (t.x * dcp0.x + t.y * dcp1.x + t.z * dcp2.x - l * drn.x + dray.x * l) / nl;
				const float dpy = (t.x * dcp0.y + t.y * dcp1.y + t.z * dcp2.y - l * drn.y + dray.y * l) / nl;
				const V3 dp3 = {dpx, dpy, 0.f};
				const float dL_dnl = (-dcp0.x * cp0.x - dcp0.y * cp0.y - dcp1.x * cp1.x - dcp1.y * cp1.y - dcp2.x * cp2.x - dcp2.y * cp2.y -
				                      drn.x * rn.x - drn.y * rn.y - dray.x * ray_plane.x - dray.y * ray_plane.y) / nl;
				const float tmp = dpx * plane0 + dpy * plane1;
				const V3 W_uvh = mulcol(Wm, uvh);
				const M3 nJ_inv_T = transpose(nJ_inv);
				M3 dL_dVrk = m3(0, 0, 0, 0, 0, 0, 0, 0, 0);
				if (si.well) {
					// -outer(Vrk_inv W uvh, (Vrk_inv / vb) (W uvh (-tmp) + W nJ_inv^T dplane))      (backward.cu:334)
					M3 Vs;
					Vs.c[0] = Vrk_inv.c[0] / clamp_vb; Vs.c[1] = Vrk_inv.c[1] / clamp_vb; Vs.c[2] = Vrk_inv.c[2] / clamp_vb;
					const V3 rhs = W_uvh * (-tmp) + mulcol(Wm * nJ_inv_T, dp3);
					const M3 o = outer(mulcol(Vrk_inv, W_uvh), mulcol(Vs, rhs));
					dL_dVrk.c[0] = V3{-o.c[0].x, -o.c[0].y, -o.c[0].z};
					dL_dVrk.c[1] = V3{-o.c[1].x, -o.c[1].y, -o.c[1].z};
					dL_dVrk.c[2] = V3{-o.c[2].x, -o.c[2].y, -o.c[2].z};
				} else {
					// rank-1 branch: through the smallest eigenvector (backward.cu:336-350)
					const float dL_dvb = -tmp / clamp_vb;
					const V3 nji = mulcol(nJ_inv_T, V3{dpx / clamp_vb, dpy / clamp_vb, 0.f});
					const M3 dVi = outer(W_uvh, W_uvh * dL_dvb + mulcol(Wm, nji));
					const M3 dViT = transpose(dVi);
					M3 sym;
					sym.c[0] = dVi.c[0] + dViT.c[0]; sym.c[1] = dVi.c[1] + dViT.c[1]; sym.c[2] = dVi.c[2] + dViT.c[2];
					const V3 emin = si.min_id == 0 ? si.E.c[0] : (si.min_id == 1 ? si.E.c[1] : si.E.c[2]);
					const V3 dLdv = mulcol(sym, emin);
#pragma unroll
					for (int j = 0; j < 3; j++) {
						if (j != si.min_id) {
							const float scale = dot3(si.E.c[j], dLdv) / min(si.lam_min - si.lam[j], -0.0000001f);
							const M3 o = outer(si.E.c[j] * scale, emin);
							dL_dVrk.c[0] = dL_dVrk.c[0] + o.c[0]; dL_dVrk.c[1] = dL_dVrk.c[1] + o.c[1]; dL_dVrk.c[2] = dL_dVrk.c[2] + o.c[2];
						}
					}
				}
				dVrk[0] = at(dL_dVrk, 0, 0);
				dVrk[3] = at(dL_dVrk, 1, 1);
				dVrk[5] = at(dL_dVrk, 2, 2);
				dVrk[1] = at(dL_dVrk, 0, 1) + at(dL_dVrk, 1, 0);
				dVrk[2] = at(dL_dVrk, 0, 2) + at(dL_dVrk, 2, 0);
				dVrk[4] = at(dL_dVrk, 1, 2) + at(dL_dVrk, 2, 1);
				// dL_duvh = 2(-tmp) q + (cov_cam_inv / vb) nJ_inv^T dplane      (backward.cu:353)
				M3 Cs;
				Cs.c[0] = cov_cam_inv.c[0] / clamp_vb; Cs.c[1] = cov_cam_inv.c[1] / clamp_vb; Cs.c[2] = cov_cam_inv.c[2] / clamp_vb;
				const V3 dL_duvh = qv * (2 * (-tmp)) + mulcol(Cs * nJ_inv_T, dp3);
				// dL_dnJ_inv = outer(dplane, q): [c][r] = dp_r q_c
				const float nji01 = dpy * qv.x, nji10 = dpx * qv.y, nji11 = dpy * qv.y, nji00 = dpx * qv.x, nji20 = dpx * qv.z, nji21 = dpy * qv.z;
				dL_du = dL_dnl * 2 * txtz + dL_duvh.x + (nji01 + nji10) * (-tytz) + 2 * nji11 * txtz - nji20 +
				        (dcp0.y * t.y + dcp1.x * t.y + dcp1.y * (-2 * t.x)) / nl;
				dL_dv = dL_dnl * 2 * tytz + dL_duvh.y + (nji01 + nji10) * (-txtz) + 2 * nji00 * tytz - nji21 +
				        (dcp0.x * (-2 * t.y) + dcp0.y * t.x + dcp1.x * t.x) / nl;
			} else {
				dcn = V3{0, 0, 0};
				rn = V3{0, 0, 0};
			}
		}

		// ---- mip-coefficient and conic backward (backward.cu:367-431) ----
		// fixed mode reads the true opacity*coef that forward stored in the render record (slot 5)
		const float combined_opacity = fix_mip ? g.records[(size_t)idx * rec_floats(p.coord) + 5] : dL_dconic.z;
		const float opacity = combined_opacity / (coef + 1e-6);
		const float dL_dcoef = dL_dopacity * opacity;
		const float dL_dsqrtcoef = dL_dcoef * 0.5 * 1. / (coef + 1e-6);
		const float dL_ddet0 = dL_dsqrtcoef / (det_1 + 1e-6);
		const float dL_ddet1 = dL_dsqrtcoef * det_0 * (-1.f / (det_1 * det_1 + 1e-6));
		const float dcoef_da = dL_ddet0 * c11 + dL_ddet1 * (c11 + ks);
		const float dcoef_db = dL_ddet0 * (-2. * c01) + dL_ddet1 * (-2. * c01);
		const float dcoef_dc = dL_ddet0 * c00 + dL_ddet1 * (c00 + ks);
		const float a = c00 + ks, b = c01, c = c11 + ks;
		const float denom = a * c - b * b;
		float dL_da = 0, dL_db = 0, dL_dc = 0;
		const float denom2inv = 1.0f / ((denom * denom) + 0.0000001f);
#define TT(col, row) at(T, col, row)
#define VV(col, row) at(Vrk, col, row)
		if (denom2inv != 0) {
			dL_da = denom2inv * (-c * c * dL_dconic.x + 2 * b * c * dL_dconic.y + (denom - a * c) * dL_dconic.z);
			dL_dc = denom2inv * (-a * a * dL_dconic.z + 2 * a * b * dL_dconic.y + (denom - a * c) * dL_dconic.x);
			dL_db = denom2inv * 2 * (b * c * dL_dconic.x - (denom + 2 * b * b) * dL_dconic.y + a * b * dL_dconic.z);
			if (det_0 <= 1e-6 || det_1 <= 1e-6) {
				dL_dopacity = 0;
			} else {
				dL_da += dcoef_da;
				dL_dc += dcoef_dc;
				dL_db += dcoef_db;
				dL_dopacity = dL_dopacity * coef;
			}
			o_cov[0] = (TT(0, 0) * TT(0, 0) * dL_da + TT(0, 0) * TT(1, 0) * dL_db + TT(1, 0) * TT(1, 0) * dL_dc);
			o_cov[3] = (TT(0, 1) * TT(0, 1) * dL_da + TT(0, 1) * TT(1, 1) * dL_db + TT(1, 1) * TT(1, 1) * dL_dc);
			o_cov[5] = (TT(0, 2) * TT(0, 2) * dL_da + TT(0, 2) * TT(1, 2) * dL_db + TT(1, 2) * TT(1, 2) * dL_dc);
			o_cov[1] = 2 * TT(0, 0) * TT(0, 1) * dL_da + (TT(0, 0) * TT(1, 1) + TT(0, 1) * TT(1, 0)) * dL_db + 2 * TT(1, 0) * TT(1, 1) * dL_dc;
			o_cov[2] = 2 * TT(0, 0) * TT(0, 2) * dL_da + (TT(0, 0) * TT(1, 2) + TT(0, 2) * TT(1, 0)) * dL_db + 2 * TT(1, 0) * TT(1, 2) * dL_dc;
			o_cov[4] = 2 * TT(0, 2) * TT(0, 1) * dL_da + (TT(0, 1) * TT(1, 2) + TT(0, 2) * TT(1, 1)) * dL_db + 2 * TT(1, 1) * TT(1, 2) * dL_dc;
		}
#pragma unroll
		for (int i = 0; i < 6; i++) o_cov[i] += dVrk[i];
		o_opacity = dL_dopacity;

		// ---- T -> J -> t (backward.cu:433-477) ----
		const float dL_dT00 = 2 * (TT(0, 0) * VV(0, 0) + TT(0, 1) * VV(0, 1) + TT(0, 2) * VV(0, 2)) * dL_da +
		                      (TT(1, 0) * VV(0, 0) + TT(1, 1) * VV(0, 1) + TT(1, 2) * VV(0, 2)) * dL_db;
		const float dL_dT01 = 2 * (TT(0, 0) * VV(1, 0) + TT(0, 1) * VV(1, 1) + TT(0, 2) * VV(1, 2)) * dL_da +
		                      (TT(1, 0) * VV(1, 0) + TT(1, 1) * VV(1, 1) + TT(1, 2) * VV(1, 2)) * dL_db;
		const float dL_dT02 = 2 * (TT(0, 0) * VV(2, 0) + TT(0, 1) * VV(2, 1) + TT(0, 2) * VV(2, 2)) * dL_da +
		                      (TT(1, 0) * VV(2, 0) + TT(1, 1) * VV(2, 1) + TT(1, 2) * VV(2, 2)) * dL_db;
		const float dL_dT10 = 2 * (TT(1, 0) * VV(0, 0) + TT(1, 1) * VV(0, 1) + TT(1, 2) * VV(0, 2)) * dL_dc +
		                      (TT(0, 0) * VV(0, 0) + TT(0, 1) * VV(0, 1) + TT(0, 2) * VV(0, 2)) * dL_db;
		const float dL_dT11 = 2 * (TT(1, 0) * VV(1, 0) + TT(1, 1) * VV(1, 1) + TT(1, 2) * VV(1, 2)) * dL_dc +
		                      (TT(0, 0) * VV(1, 0) + TT(0, 1) * VV(1, 1) + TT(0, 2) * VV(1, 2)) * dL_db;
		const float dL_dT12 = 2 * (TT(1, 0) * VV(2, 0) + TT(1, 1) * VV(2, 1) + TT(1, 2) * VV(2, 2)) * dL_dc +
		                      (TT(0, 0) * VV(2, 0) + TT(0, 1) * VV(2, 1) + TT(0, 2) * VV(2, 2)) * dL_db;
#undef TT
#undef VV
		const float dL_dJ00 = at(Wm, 0, 0) * dL_dT00 + at(Wm, 0, 1) * dL_dT01 + at(Wm, 0, 2) * dL_dT02;
		const float dL_dJ02 = at(Wm, 2, 0) * dL_dT00 + at(Wm, 2, 1) * dL_dT01 + at(Wm, 2, 2) * dL_dT02;
		const float dL_dJ11 = at(Wm, 1, 0) * dL_dT10 + at(Wm, 1, 1) * dL_dT11 + at(Wm, 1, 2) * dL_dT12;
		const float dL_dJ12 = at(Wm, 2, 0) * dL_dT10 + at(Wm, 2, 1) * dL_dT11 + at(Wm, 2, 2) * dL_dT12;

		const float tz = 1.f / t.z, tz2 = tz * tz, tz3 = tz2 * tz;
		const float l3 = l * l * l;
		// dL_dnJ[c][r] = dcn_r * rn_c
		const float nJ02 = dcn.z * rn.x, nJ12 = dcn.z * rn.y, nJ20 = dcn.x * rn.z, nJ21 = dcn.y * rn.z, nJ22 = dcn.z * rn.z;
		const float nJ00 = dcn.x * rn.x, nJ11 = dcn.y * rn.y;
		const float dL_dtx = x_grad_mul * (-h_x * tz2 * dL_dJ02 + dL_du * tz - nJ02 * tz2 + nJ20 * (1 / l - t.x * t.x / l3) + nJ21 * (-t.x * t.y / l3) +
		                                   nJ22 * (-t.x * t.z / l3) + (dcp0.x * plane0 + dcp0.y * plane1 + dcp2.x) / nl + dL_dl * t.x / l);
		const float dL_dty = y_grad_mul * (-h_y * tz2 * dL_dJ12 + dL_dv * tz - nJ12 * tz2 + nJ20 * (-t.x * t.y / l3) + nJ21 * (1 / l - t.y * t.y / l3) +
		                                   nJ22 * (-t.y * t.z / l3) + (dcp1.x * plane0 + dcp1.y * plane1 + dcp2.y) / nl + dL_dl * t.y / l);
		const float dL_dtz = -h_x * tz2 * dL_dJ00 - h_y * tz2 * dL_dJ11 + (2 * h_x * t.x) * tz3 * dL_dJ02 + (2 * h_y * t.y) * tz3 * dL_dJ12 -
		                     (dL_du * t.x + dL_dv * t.y) * tz2 + (nJ00 + nJ11) * (-tz2) + nJ02 * (2 * t.x * tz3) + nJ12 * (2 * t.y * tz3) +
		                     (nJ20 * t.x + nJ21 * t.y) * (-t.z / l3) + nJ22 * (1 / l - t.z * t.z / l3) +
		                     (dcp0.x * (-(v2 + 1)) + dcp0.y * uv + dcp1.x * uv + dcp1.y * (-(u2 + 1)) + dcp2.x * plane0 + dcp2.y * plane1) / nl +
		                     dL_dl * t.z / l;
		float3 dL_dmean = xformvec4x3T(float3{dL_dtx, dL_dty, dL_dtz}, V);

		// ---- screen-space mean, ray length and view-point terms (backward.cu:587-619) ----
		{
			const float* proj = p.projmatrix;
			const float4 m_hom = xform4x4(mean, proj);
			const float m_w = 1.0f / (m_hom.w + 0.0000001f);
			const float mul1 = (proj[0] * mean.x + proj[4] * mean.y + proj[8] * mean.z + proj[12]) * m_w * m_w;
			const float mul2 = (proj[1] * mean.x + proj[5] * mean.y + proj[9] * mean.z + proj[13]) * m_w * m_w;
			float3 d1;
			d1.x = (proj[0] * m_w - proj[3] * mul1) * dL_dmean2D.x + (proj[1] * m_w - proj[3] * mul2) * dL_dmean2D.y;
			d1.y = (proj[4] * m_w - proj[7] * mul1) * dL_dmean2D.x + (proj[5] * m_w - proj[7] * mul2) * dL_dmean2D.y;
			d1.z = (proj[8] * m_w - proj[11] * mul1) * dL_dmean2D.x + (proj[9] * m_w - proj[11] * mul2) * dL_dmean2D.y;
			const float3 m_view = xform4x3(mean, V);
			const float tl = sqrt(m_view.x * m_view.x + m_view.y * m_view.y + m_view.z * m_view.z);
			const float3 d2 = xformvec4x3T(float3{dL_dview_point.x + m_view.x / tl * dL_dts, dL_dview_point.y + m_view.y / tl * dL_dts,
			                                      dL_dview_point.z + m_view.z / tl * dL_dts}, V);
			dL_dmean.x += d1.x + d2.x;
			dL_dmean.y += d1.y + d2.y;
			dL_dmean.z += d1.z + d2.z;
		}

		// (the SH term of dL_dmean and dL_dsh are produced by sh_backward_rows_kernel, launched right after this kernel)
		o_mean3D[0] = dL_dmean.x; o_mean3D[1] = dL_dmean.y; o_mean3D[2] = dL_dmean.z;

		// ---- covariance -> scale / rotation (backward.cu:492-555) ----
		if (from_scales) {
			// M = S * Rg (glm), dL_dM = 2 M dL_dSigma ; dL_dMt = transpose(dL_dM)
			M3 S = m3(s_mod.x, 0.f, 0.f, 0.f, s_mod.y, 0.f, 0.f, 0.f, s_mod.z);
			M3 Mm = S * Rg;
			M3 dSig = m3(o_cov[0], 0.5f * o_cov[1], 0.5f * o_cov[2], 0.5f * o_cov[1], o_cov[3], 0.5f * o_cov[4], 0.5f * o_cov[2], 0.5f * o_cov[4], o_cov[5]);
			M3 dM = Mm * dSig;
			dM.c[0] = dM.c[0] * 2.0f; dM.c[1] = dM.c[1] * 2.0f; dM.c[2] = dM.c[2] * 2.0f;
			M3 Rt = transpose(Rg);
			M3 dMt = transpose(dM);
			o_scale[0] = dot3(Rt.c[0], dMt.c[0]);
			o_scale[1] = dot3(Rt.c[1], dMt.c[1]);
			o_scale[2] = dot3(Rt.c[2], dMt.c[2]);
			dMt.c[0] = dMt.c[0] * s_mod.x;
			dMt.c[1] = dMt.c[1] * s_mod.y;
			dMt.c[2] = dMt.c[2] * s_mod.z;
			const float r = q.x, x = q.y, y = q.z, z = q.w;
#define D(c_, r_) at(dMt, c_, r_)
			o_rot[0] = 2 * z * (D(0, 1) - D(1, 0)) + 2 * y * (D(2, 0) - D(0, 2)) + 2 * x * (D(1, 2) - D(2, 1));
			o_rot[1] = 2 * y * (D(1, 0) + D(0, 1)) + 2 * z * (D(2, 0) + D(0, 2)) + 2 * r * (D(1, 2) - D(2, 1)) - 4 * x * (D(2, 2) + D(1, 1));
			o_rot[2] = 2 * x * (D(1, 0) + D(0, 1)) + 2 * r * (D(2, 0) - D(0, 2)) + 2 * z * (D(1, 2) + D(2, 1)) - 4 * y * (D(2, 2) + D(0, 0));
			o_rot[3] = 2 * r * (D(0, 1) - D(1, 0)) + 2 * x * (D(2, 0) + D(0, 2)) + 2 * y * (D(1, 2) + D(2, 1)) - 4 * z * (D(1, 1) + D(0, 0));
#undef D
			// the reference scales dL_dscale by nothing further: d(mod*s)/ds = mod is NOT applied (backward.cu:536-539)
		}
	}

	// ---- write everything ----
#pragma unroll
	for (int i = 0; i < 3; i++) {
		out.d_means2D[3 * idx + i] = o_means2D[i];
		out.d_colors[3 * idx + i] = o_colors[i];
		out.d_means3D[3 * idx + i] = o_mean3D[i];
		out.d_scales[3 * idx + i] = o_scale[i];
	}
	out.d_opacity[idx] = o_opacity;
#pragma unroll
	for (int i = 0; i < 6; i++) out.d_cov3D[6 * idx + i] = o_cov[i];
	*reinterpret_cast<float4*>(out.d_rotations + 4 * idx) = make_float4(o_rot[0], o_rot[1], o_rot[2], o_rot[3]);
}

// One thread per LISTED Gaussian (rendered and with a non-zero accumulator row); the outputs of all other rows were zero-filled
// before.  In a dense scene most rendered splats are occluded in any one view (C2: 84 %, C3: 92 % of the visible ones receive
// nothing), and a warp of a thread-per-Gaussian kernel would run the whole chain if ANY of its 32 rows needed it.
__global__ void __launch_bounds__(128, 4) preprocess_backward_rows_kernel(FwdParams p, GeomView g, const int* __restrict__ radii,
                                                                        const float* __restrict__ grad_accum, ParamGradOut out, int fix_mip,
                                                                        const uint32_t* __restrict__ list, const uint32_t* __restrict__ count) {
	const int n = (int)*count;
	for (int l = blockIdx.x * blockDim.x + threadIdx.x; l < n; l += gridDim.x * blockDim.x)
		preprocess_backward_row(p, g, radii, grad_accum, out, fix_mip, (int)list[l]);
}

// rows that need work: rendered and any non-zero (or NaN) entry in the accumulator row.  A warp owns 32 consecutive rows and reads them
// as one contiguous block (lane-major float4, RQ passes of 512 bytes), folds the quarters of a row with a ballot, and appends the
// surviving rows with ONE atomic per warp.
template <int RQ>
__global__ void __launch_bounds__(256) nonzero_rows_kernel(int P, const int* __restrict__ radii, const float4* __restrict__ grad_accum,
                                                            uint32_t* __restrict__ list, uint32_t* __restrict__ count) {
	const int lane = threadIdx.x & 31;
	const int row0 = (blockIdx.x * blockDim.x + threadIdx.x) - lane;  // first of this warp's 32 rows
	if (row0 >= P) return;
	const int idx = row0 + lane;
	const bool vis = idx < P && radii[idx] > 0;
	const size_t n4 = (size_t)P * RQ;
	unsigned rows_nz = 0;  // bit r: row row0 + r has a non-zero entry
#pragma unroll
	for (int k = 0; k < RQ; k++) {
		const size_t e = (size_t)row0 * RQ + (size_t)k * 32 + lane;  // float4 index: row (k*32+lane)/RQ, quarter (k*32+lane)%RQ
		float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
		if (e < n4) v = grad_accum[e];
		const bool nzq = !(v.x == 0.f) || !(v.y == 0.f) || !(v.z == 0.f) || !(v.w == 0.f);
		unsigned b = __ballot_sync(0xffffffffu, nzq);  // bit j: float4 k*32+j
		// fold groups of RQ bits into one bit per row
#pragma unroll
		for (int sft = 1; sft < RQ; sft <<= 1) b |= b >> sft;
		// rows covered by this pass: (k*32)/RQ ... ; pick bit (r*RQ) of b for the r-th of them
		constexpr int rows_per_pass = 32 / RQ;
#pragma unroll
		for (int r = 0; r < rows_per_pass; r++)
			if ((b >> (r * RQ)) & 1u) rows_nz |= 1u << (k * rows_per_pass + r);
	}
	const unsigned keep = rows_nz & __ballot_sync(0xffffffffu, vis);
	if (keep == 0) return;
	uint32_t base = 0;
	if (lane == 0) base = atomicAdd(count, (uint32_t)__popc(keep));
	base = __shfl_sync(0xffffffffu, base, 0);
	if ((keep >> lane) & 1u) list[base + __popc(keep & ((1u << lane) - 1u))] = (uint32_t)idx;
}

// ---- SH backward (backward.cu:21-140) ----------------------------------------------------------------------------------
// dL_dsh of every listed Gaussian, and the view-direction term added to dL_dmeans3D (third part of the mean gradient,
// backward.cu:131-139).  Each lane works on its coefficient row in a shared-memory scratch row (row stride padded to an odd
// number of floats: conflict-free).
constexpr int SH_WARPS = 8;

// SH backward of ONE Gaussian whose [M,3] coefficient row sits at `sh` (shared memory): the row is overwritten with dL_dsh and the
// view-direction term is added to dL_dmeans3D (backward.cu:21-140).
__device__ __forceinline__ void sh_backward_row(float* sh, int idx, int D, int M, const float* __restrict__ means3D, const float* __restrict__ cam_pos,
                                                const uint8_t* __restrict__ clamped, const float* __restrict__ grad_accum, int GF,
                                                float* __restrict__ d_means3D) {
	const float3 mean = {means3D[3 * idx], means3D[3 * idx + 1], means3D[3 * idx + 2]};
	const float3 campos = {cam_pos[0], cam_pos[1], cam_pos[2]};
	const float3 dir_orig = {mean.x - campos.x, mean.y - campos.y, mean.z - campos.z};
	const float dlen = sqrtf(dir_orig.x * dir_orig.x + dir_orig.y * dir_orig.y + dir_orig.z * dir_orig.z);
	const float x = dir_orig.x / dlen, y = dir_orig.y / dlen, z = dir_orig.z / dlen;
	const uint8_t cb = clamped[idx];
	const float* ga = grad_accum + (size_t)idx * GF + G_COL;
	const float dRGB[3] = {(cb & 1) ? 0.f : ga[0], (cb & 2) ? 0.f : ga[1], (cb & 4) ? 0.f : ga[2]};
	const int deg = D;
	float basis[16];
	float ddx[16], ddy[16], ddz[16];  // d(basis_k)/d(dir)
#pragma unroll
	for (int k = 0; k < 16; k++) { basis[k] = 0.f; ddx[k] = 0.f; ddy[k] = 0.f; ddz[k] = 0.f; }
	basis[0] = kSH0;
	if (deg > 0) {
		basis[1] = -kSH1 * y; basis[2] = kSH1 * z; basis[3] = -kSH1 * x;
		ddx[3] = -kSH1; ddy[1] = -kSH1; ddz[2] = kSH1;
		if (deg > 1) {
			const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
			basis[4] = kSH2[0] * xy; basis[5] = kSH2[1] * yz; basis[6] = kSH2[2] * (2.f * zz - xx - yy);
			basis[7] = kSH2[3] * xz; basis[8] = kSH2[4] * (xx - yy);
			ddx[4] = kSH2[0] * y; ddx[6] = kSH2[2] * 2.f * -x; ddx[7] = kSH2[3] * z; ddx[8] = kSH2[4] * 2.f * x;
			ddy[4] = kSH2[0] * x; ddy[5] = kSH2[1] * z; ddy[6] = kSH2[2] * 2.f * -y; ddy[8] = kSH2[4] * 2.f * -y;
			ddz[5] = kSH2[1] * y; ddz[6] = kSH2[2] * 2.f * 2.f * z; ddz[7] = kSH2[3] * x;
			if (deg > 2) {
				basis[9] = kSH3[0] * y * (3.f * xx - yy); basis[10] = kSH3[1] * xy * z;
				basis[11] = kSH3[2] * y * (4.f * zz - xx - yy); basis[12] = kSH3[3] * z * (2.f * zz - 3.f * xx - 3.f * yy);
				basis[13] = kSH3[4] * x * (4.f * zz - xx - yy); basis[14] = kSH3[5] * z * (xx - yy);
				basis[15] = kSH3[6] * x * (xx - 3.f * yy);
				ddx[9] = kSH3[0] * 3.f * 2.f * xy; ddx[10] = kSH3[1] * yz; ddx[11] = kSH3[2] * -2.f * xy; ddx[12] = kSH3[3] * -3.f * 2.f * xz;
				ddx[13] = kSH3[4] * (-3.f * xx + 4.f * zz - yy); ddx[14] = kSH3[5] * 2.f * xz; ddx[15] = kSH3[6] * 3.f * (xx - yy);
				ddy[9] = kSH3[0] * 3.f * (xx - yy); ddy[10] = kSH3[1] * xz; ddy[11] = kSH3[2] * (-3.f * yy + 4.f * zz - xx);
				ddy[12] = kSH3[3] * -3.f * 2.f * yz; ddy[13] = kSH3[4] * -2.f * xy; ddy[14] = kSH3[5] * -2.f * yz; ddy[15] = kSH3[6] * -3.f * 2.f * xy;
				ddz[10] = kSH3[1] * xy; ddz[11] = kSH3[2] * 4.f * 2.f * yz; ddz[12] = kSH3[3] * 3.f * (2.f * zz - xx - yy);
				ddz[13] = kSH3[4] * 4.f * 2.f * xz; ddz[14] = kSH3[5] * (xx - yy);
			}
		}
	}
	const int ncoef = (deg + 1) * (deg + 1);
	float3 dL_ddir = {0.f, 0.f, 0.f};
#pragma unroll
	for (int k = 0; k < 16; k++) {
		if (k < M) {
			float o0 = 0.f, o1 = 0.f, o2 = 0.f;
			if (k < ncoef) {
				o0 = basis[k] * dRGB[0]; o1 = basis[k] * dRGB[1]; o2 = basis[k] * dRGB[2];
				if (k > 0) {
					const float sd = sh[3 * k] * dRGB[0] + sh[3 * k + 1] * dRGB[1] + sh[3 * k + 2] * dRGB[2];
					dL_ddir.x += ddx[k] * sd;
					dL_ddir.y += ddy[k] * sd;
					dL_ddir.z += ddz[k] * sd;
				}
			}
			sh[3 * k] = o0; sh[3 * k + 1] = o1; sh[3 * k + 2] = o2;
		}
	}
	// through the normalisation of the view direction (auxiliary.h:123-133)
	const float sum2 = dir_orig.x * dir_orig.x + dir_orig.y * dir_orig.y + dir_orig.z * dir_orig.z;
	const float invsum32 = 1.0f / sqrt(sum2 * sum2 * sum2);
	float* dm = d_means3D + 3 * idx;
	dm[0] += ((+sum2 - dir_orig.x * dir_orig.x) * dL_ddir.x - dir_orig.y * dir_orig.x * dL_ddir.y - dir_orig.z * dir_orig.x * dL_ddir.z) * invsum32;
	dm[1] += (-dir_orig.x * dir_orig.y * dL_ddir.x + (sum2 - dir_orig.y * dir_orig.y) * dL_ddir.y - dir_orig.z * dir_orig.y * dL_ddir.z) * invsum32;
	dm[2] += (-dir_orig.x * dir_orig.z * dL_ddir.x - dir_orig.y * dir_orig.z * dL_ddir.y + (sum2 - dir_orig.z * dir_orig.z) * dL_ddir.z) * invsum32;
}

// Lane = one LISTED Gaussian.  The rows are scattered in memory, so every lane fetches its own coefficient row (12*M contiguous bytes:
// twelve independent 128-bit loads in flight when the layout allows) into its shared-memory scratch row, works on it in place and
// stores dL_dsh back the same way; all other rows of dL_dsh were zero-filled.
__global__ void __launch_bounds__(SH_WARPS * 32) sh_backward_rows_kernel(int D, int M, const float* __restrict__ means3D, const float* __restrict__ cam_pos,
                                                                          const float* __restrict__ shs, const float* __restrict__ shs_rest,
                                                                          const uint8_t* __restrict__ clamped, const float* __restrict__ grad_accum, int GF,
                                                                          float* __restrict__ d_sh, float* __restrict__ d_sh_rest,
                                                                          float* __restrict__ d_means3D, const uint32_t* __restrict__ list,
                                                                          const uint32_t* __restrict__ count) {
	extern __shared__ float s_sh[];
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const int row = 3 * M, stride = row | 1;
	float* sh = s_sh + ((size_t)warp * 32 + lane) * stride;
	const bool split = shs_rest != nullptr;
	const bool vec = !split && (row & 3) == 0 && (reinterpret_cast<uintptr_t>(shs) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_sh) & 15) == 0;
	const int n = (int)*count;
	for (int l = blockIdx.x * blockDim.x + threadIdx.x; l < n; l += gridDim.x * blockDim.x) {
		const int rid = (int)list[l];
		const uint8_t cb = clamped[rid];
		const float* ga = grad_accum + (size_t)rid * GF + G_COL;
		// a zero colour gradient (after the clamp mask) leaves dL_dsh = 0 and no view-direction term: nothing to read or write
		if (!((!(cb & 1) && !(ga[0] == 0.f)) || (!(cb & 2) && !(ga[1] == 0.f)) || (!(cb & 4) && !(ga[2] == 0.f)))) continue;
		if (vec) {
			const float4* src = reinterpret_cast<const float4*>(shs + (size_t)rid * row);
			float4 v[12];
#pragma unroll
			for (int q = 0; q < 12; q++)
				if (4 * q < row) v[q] = __ldg(src + q);
#pragma unroll
			for (int q = 0; q < 12; q++)
				if (4 * q < row) { sh[4 * q] = v[q].x; sh[4 * q + 1] = v[q].y; sh[4 * q + 2] = v[q].z; sh[4 * q + 3] = v[q].w; }
		} else if (!split) {
			const float* src = shs + (size_t)rid * row;
			for (int e = 0; e < row; e++) sh[e] = __ldg(src + e);
		} else {
			const float* s0 = shs + (size_t)rid * 3;
			const float* s1 = shs_rest + (size_t)rid * (row - 3);
			sh[0] = __ldg(s0); sh[1] = __ldg(s0 + 1); sh[2] = __ldg(s0 + 2);
			for (int e = 0; e < row - 3; e++) sh[3 + e] = __ldg(s1 + e);
		}
		sh_backward_row(sh, rid, D, M, means3D, cam_pos, clamped, grad_accum, GF, d_means3D);
		if (vec) {
			float4* dst = reinterpret_cast<float4*>(d_sh + (size_t)rid * row);
#pragma unroll
			for (int q = 0; q < 12; q++)
				if (4 * q < row) dst[q] = make_float4(sh[4 * q], sh[4 * q + 1], sh[4 * q + 2], sh[4 * q + 3]);
		} else if (!split) {
			float* dst = d_sh + (size_t)rid * row;
			for (int e = 0; e < row; e++) dst[e] = sh[e];
		} else {
			float* d0 = d_sh + (size_t)rid * 3;
			float* d1 = d_sh_rest + (size_t)rid * (row - 3);
			d0[0] = sh[0]; d0[1] = sh[1]; d0[2] = sh[2];
			for (int e = 0; e < row - 3; e++) d1[e] = sh[3 + e];
		}
	}
}

// zero-fill of the nine dense gradient tensors (what the row kernels do not write).  Pure HBM writes: rgs_backward issues it on
// a side stream so that it runs underneath the issue-bound backward blend.
void launch_backward_zero_fill(const FwdParams& p, ParamGradOut out, cudaStream_t s) {
	const size_t P = (size_t)p.P;
	const bool has_sh = p.shs != nullptr && out.d_sh != nullptr && p.M > 0;
	const bool split = p.shs_rest != nullptr;
	cudaMemsetAsync(out.d_means2D, 0, P * 3 * sizeof(float), s);
	cudaMemsetAsync(out.d_colors, 0, P * 3 * sizeof(float), s);
	cudaMemsetAsync(out.d_opacity, 0, P * sizeof(float), s);
	cudaMemsetAsync(out.d_means3D, 0, P * 3 * sizeof(float), s);
	cudaMemsetAsync(out.d_cov3D, 0, P * 6 * sizeof(float), s);
	cudaMemsetAsync(out.d_scales, 0, P * 3 * sizeof(float), s);
	cudaMemsetAsync(out.d_rotations, 0, P * 4 * sizeof(float), s);
	if (has_sh) {
		cudaMemsetAsync(out.d_sh, 0, P * (split ? 3 : 3 * p.M) * sizeof(float), s);
		if (split && out.d_sh_rest != nullptr) cudaMemsetAsync(out.d_sh_rest, 0, P * (3 * p.M - 3) * sizeof(float), s);
	}
}

void launch_preprocess_backward(const FwdParams& p, GeomView g, const int* radii, const float* grad_accum, ParamGradOut out, cudaStream_t s,
                                bool prefilled) {
	static const int fix_mip = getenv("RGS_FIX_MIP_GRADIENT") != nullptr && atoi(getenv("RGS_FIX_MIP_GRADIENT")) != 0;
	const bool has_sh = p.shs != nullptr && out.d_sh != nullptr && p.M > 0;
	// zero-fill the outputs (memsets run at HBM write speed), list the rows that received anything, run the chains on those
	if (!prefilled) launch_backward_zero_fill(p, out, s);
	uint32_t* list = g.bwd_rows;
	uint32_t* count = g.bwd_row_count;
	cudaMemsetAsync(count, 0, sizeof(uint32_t), s);
	const int GF = grad_floats(p.coord);
	if (GF == GRAD_FLOATS_BASE)
		nonzero_rows_kernel<GRAD_FLOATS_BASE / 4><<<(p.P + 255) / 256, 256, 0, s>>>(p.P, radii, reinterpret_cast<const float4*>(grad_accum), list, count);
	else
		nonzero_rows_kernel<GRAD_FLOATS_COORD / 4><<<(p.P + 255) / 256, 256, 0, s>>>(p.P, radii, reinterpret_cast<const float4*>(grad_accum), list, count);
	// the list length stays on the device (no host sync): grids sized for "every row listed", CTAs beyond the list leave at once
	const int sms = 148;
	const int rows_grid = min((p.P + 127) / 128, sms * 16);
	preprocess_backward_rows_kernel<<<rows_grid, 128, 0, s>>>(p, g, radii, grad_accum, out, fix_mip, list, count);
	count_launch(2 + 8 + (has_sh ? 1 : 0));
	if (has_sh) {
		const size_t smem = (size_t)SH_WARPS * 32 * ((3 * p.M) | 1) * sizeof(float);
		static size_t configured[64] = {};
		if (smem > 48 * 1024) ensure_dynamic_smem(sh_backward_rows_kernel, smem, configured);
		const int sh_grid = min((p.P + SH_WARPS * 32 - 1) / (SH_WARPS * 32), sms * 8);
		sh_backward_rows_kernel<<<sh_grid, SH_WARPS * 32, smem, s>>>(p.D, p.M, p.means3D, p.cam_pos, p.shs, p.shs_rest, g.clamped, grad_accum, GF, out.d_sh,
		                                                            out.d_sh_rest, out.d_means3D, list, count);
		count_launch();
	}
}

}  // namespace rgs
