// rgs_binning.cu -- per-tile instance counts and ranges, (tile | depth) key sort, tile-bucket binning.
//
// Replaces cub::DeviceScan::InclusiveSum + duplicateWithKeys + cub::DeviceRadixSort::SortPairs +
// identifyTileRanges (reference: cuda_rasterizer/rasterizer_impl.cu:350, 70-111, 373-381, 151-173).
//
// Contract kept bit-exact with the reference: key = (tile_id << 32) | float_bits(view z), value = Gaussian
// index, and the order is the reference's stable sort of instances emitted in ascending Gaussian index -- so
// equal (tile, depth) pairs stay in ascending Gaussian index.
#include "rgs_common.cuh"

namespace rgs {

// =====================================================================================================================
// Tile-bucket binning.
//
// The reference sorts all R instances globally on 45-bit (tile | depth) keys: six 8-bit onesweep passes, each
// reading and writing 12 B per instance.  The same total order is (tile, depth bits, Gaussian index), so it is
// produced here with one bucketing step and one local sort instead:
//   1. preprocess marks every splat's tile rectangle with +1 / -1 at its four corners on a (grid_y+1) x (grid_x+1)
//      difference grid (4 red.global.add per splat, whatever the rectangle's size);
//   2. tile_scan_kernel: 2D prefix sum of that grid = instances per tile, then the exclusive scan of the T counts ->
//      ranges[tile] = [start, end), num_rendered, longest list;
//   3. scatter_kernel: every instance takes a slot inside its tile's segment (counter counted back down) and
//      stores the 64-bit local key (depth bits << 32 | Gaussian index) -- 8 B written once;
//   4. tile_sort_kernel: one CTA per tile loads its segment into shared memory, merge-sorts the 64-bit keys
//      (register network for runs of 8, then merge-path passes) and writes the ids (and the reference-format keys).
// Equal depth bits fall back to the Gaussian index through the low key half, which is exactly what the reference's
// stable sort yields (instances are emitted in ascending Gaussian index).  Global traffic: 8 B + 8 B + 4 B (+ 8 B
// for the exported keys) per instance instead of ~156 B.
// Lists longer than TILE_SORT_CAP (shared-memory capacity) are split over several CTAs: chunk sort + global merge passes (below).
// =====================================================================================================================

__global__ void __launch_bounds__(1024) tile_scan_kernel(int grid_x, int grid_y, int* __restrict__ tile_diff, uint32_t* __restrict__ tile_count,
                                                          uint2* __restrict__ ranges, uint32_t* __restrict__ chunk_base,
                                                          uint32_t* __restrict__ totals) {
	__shared__ uint32_t s_warp[32], s_warp2[32];
	__shared__ uint32_t s_max;
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const int tiles = grid_x * grid_y;
	if (tid == 0) s_max = 0;
	// phase 0: 2D prefix sum of the corner-difference grid preprocess filled -> instances per tile (exact integers).
	// One CTA, so __syncthreads orders the global accesses.
	//   rows:    a warp per row, 32 columns at a time (coalesced), inclusive shuffle scan + carry, in place;
	//   columns: the rows are cut into 32 segments (one per warp); lanes are columns (coalesced).  Each warp leaves the
	//            running sums of its segment in place and the segment totals in shared memory; after a barrier every
	//            warp adds the totals of the segments above it and writes the compact [tiles] counts.
	{
		__shared__ int s_seg[32][256];
		const int W1 = grid_x + 1;
		for (int y = warp; y < grid_y; y += 32) {
			int* row = tile_diff + (size_t)y * W1;
			int carry = 0;
			for (int x0 = 0; x0 < grid_x; x0 += 32) {
				const int x = x0 + lane;
				int v = x < grid_x ? row[x] : 0;
#pragma unroll
				for (int o = 1; o < 32; o <<= 1) {
					const int n = __shfl_up_sync(0xffffffffu, v, o);
					if (lane >= o) v += n;
				}
				v += carry;
				if (x < grid_x) row[x] = v;
				carry = __shfl_sync(0xffffffffu, v, 31);
			}
		}
		__syncthreads();
		const int rows_per = (grid_y + 31) / 32;
		const int ya = min(grid_y, warp * rows_per), yb = min(grid_y, ya + rows_per);
		for (int xb0 = 0; xb0 < grid_x; xb0 += 256) {  // column blocks of 256 (shared-memory capacity), 32 lanes at a time
			for (int x0 = xb0; x0 < min(grid_x, xb0 + 256); x0 += 32) {
				const int x = x0 + lane;
				int run = 0;
				if (x < grid_x)
					for (int y = ya; y < yb; y++) { run += tile_diff[(size_t)y * W1 + x]; tile_diff[(size_t)y * W1 + x] = run; }
				s_seg[warp][x0 - xb0 + lane] = run;
			}
			__syncthreads();
			for (int x0 = xb0; x0 < min(grid_x, xb0 + 256); x0 += 32) {
				const int x = x0 + lane;
				if (x < grid_x) {
					int off = 0;
					for (int sgm = 0; sgm < warp; sgm++) off += s_seg[sgm][x0 - xb0 + lane];
					for (int y = ya; y < yb; y++) tile_count[(size_t)y * grid_x + x] = (uint32_t)(tile_diff[(size_t)y * W1 + x] + off);
				}
			}
			__syncthreads();
		}
	}
	__syncthreads();
	// exclusive scan of the per-tile counts (and of their 32-instance chunk counts): every thread owns a run of
	// consecutive tiles -- local sums, one block scan of the 1024 partials, then the run is written out
	const int items = (tiles + 1023) / 1024;
	const int t0 = min(tiles, tid * items), t1 = min(tiles, t0 + items);
	uint32_t sum = 0, sum2 = 0, local_max = 0;
	for (int t = t0; t < t1; t++) {
		const uint32_t c = tile_count[t];
		sum += c;
		sum2 += (c + 31u) >> 5;  // 32-instance chunks of this tile (hit-mask words per pixel block)
		local_max = max(local_max, c);
	}
	uint32_t v = sum, v2 = sum2;  // inclusive warp scans
#pragma unroll
	for (int o = 1; o < 32; o <<= 1) {
		const uint32_t n = __shfl_up_sync(0xffffffffu, v, o);
		const uint32_t n2 = __shfl_up_sync(0xffffffffu, v2, o);
		if (lane >= o) { v += n; v2 += n2; }
	}
	if (lane == 31) { s_warp[warp] = v; s_warp2[warp] = v2; }
	__syncthreads();
	if (warp == 0) {
		uint32_t w = s_warp[lane], w2 = s_warp2[lane];
#pragma unroll
		for (int o = 1; o < 32; o <<= 1) {
			const uint32_t n = __shfl_up_sync(0xffffffffu, w, o);
			const uint32_t n2 = __shfl_up_sync(0xffffffffu, w2, o);
			if (lane >= o) { w += n; w2 += n2; }
		}
		s_warp[lane] = w;
		s_warp2[lane] = w2;
	}
	__syncthreads();
	uint32_t run = v - sum + (warp > 0 ? s_warp[warp - 1] : 0u);
	uint32_t run2 = v2 - sum2 + (warp > 0 ? s_warp2[warp - 1] : 0u);
	for (int t = t0; t < t1; t++) {
		const uint32_t c = tile_count[t];
		ranges[t] = c ? make_uint2(run, run + c) : make_uint2(0u, 0u);  // empty tiles stay (0,0) like the reference's memset
		chunk_base[t] = run2;
		run += c;
		run2 += (c + 31u) >> 5;
	}
#pragma unroll
	for (int o = 16; o > 0; o >>= 1) local_max = max(local_max, __shfl_xor_sync(0xffffffffu, local_max, o));
	if (lane == 0) atomicMax(&s_max, local_max);
	__syncthreads();
	if (tid == 0) { totals[0] = s_warp[31]; totals[1] = s_max; }
}

void launch_tile_scan(const FwdParams& p, ImgView img, cudaStream_t s) {
	tile_scan_kernel<<<1, 1024, 0, s>>>(p.grid_x, p.grid_y, img.tile_diff, img.tile_count, img.ranges, img.chunk_base, img.totals);
	count_launch();
}

// Scatter: every instance takes a slot inside its tile's segment and stores its 64-bit local key.
// A warp owns 32 consecutive Gaussians and emits them COOPERATIVELY: the tiles of one splat are spread over the lanes
// (lane k takes the k-th tile of the rectangle), four splats are in flight per round so that the returning atomics
// (slot = counter counted back down) of one splat overlap the key stores of the previous ones.  A thread-per-splat
// loop would serialise one ~1 us atomic round trip per tile and let a few large splats hold the whole grid.
__global__ void __launch_bounds__(256) scatter_kernel(int P, const float* __restrict__ records, int rec_f, const float* __restrict__ depths,
                                                       const uint32_t* __restrict__ tiles_touched, const int* __restrict__ radii, int grid_x, int grid_y,
                                                       int row_begin, int row_end, const uint2* __restrict__ ranges, uint32_t* __restrict__ tile_count,
                                                       uint64_t* __restrict__ local_keys) {
	const int lane = threadIdx.x & 31;
	const int idx = blockIdx.x * blockDim.x + threadIdx.x;
	int cnt = 0, x0 = 0, y0 = 0, w = 1;
	uint32_t dbits = 0;
	if (idx < P) {
		cnt = (int)tiles_touched[idx];
		if (cnt > 0) {
			const float2 xy = *reinterpret_cast<const float2*>(records + (size_t)idx * rec_f);
			uint2 rmin, rmax;
			tile_rect(xy, radii[idx], grid_x, grid_y, rmin, rmax);
			x0 = (int)rmin.x;
			w = (int)rmax.x - (int)rmin.x;
			y0 = max((int)rmin.y, row_begin);
			dbits = __float_as_uint(depths[idx]);
		}
	}
	unsigned live = __ballot_sync(0xffffffffu, cnt > 0);
	while (live) {
		int s_cnt[4], s_x0[4], s_y0[4], s_w[4], s_tile[4];
		uint32_t s_slot[4];
		uint64_t s_key[4];
		bool act[4];
#pragma unroll
		for (int u = 0; u < 4; u++) {
			act[u] = false;
			s_cnt[u] = 0;
			if (live) {
				const int src = __ffs(live) - 1;
				live &= live - 1;
				s_cnt[u] = __shfl_sync(0xffffffffu, cnt, src);
				s_x0[u] = __shfl_sync(0xffffffffu, x0, src);
				s_y0[u] = __shfl_sync(0xffffffffu, y0, src);
				s_w[u] = __shfl_sync(0xffffffffu, w, src);
				const uint32_t db = __shfl_sync(0xffffffffu, dbits, src);
				s_key[u] = ((uint64_t)db << 32) | (uint32_t)(idx - lane + src);
				if (lane < s_cnt[u]) {
					const int ry = lane / s_w[u], rx = lane - ry * s_w[u];
					s_tile[u] = (s_y0[u] + ry) * grid_x + s_x0[u] + rx;
					s_slot[u] = atomicSub(tile_count + s_tile[u], 1u) - 1u;
					act[u] = true;
				}
			}
		}
#pragma unroll
		for (int u = 0; u < 4; u++)
			if (act[u]) local_keys[ranges[s_tile[u]].x + s_slot[u]] = s_key[u];
		// splats covering more than 32 tiles: remaining tiles, 32 per round
#pragma unroll
		for (int u = 0; u < 4; u++) {
			for (int k = lane + 32; k < s_cnt[u]; k += 32) {
				const int ry = k / s_w[u], rx = k - ry * s_w[u];
				const int t = (s_y0[u] + ry) * grid_x + s_x0[u] + rx;
				const uint32_t slot = atomicSub(tile_count + t, 1u) - 1u;
				local_keys[ranges[t].x + slot] = s_key[u];
			}
		}
	}
}

// ---- per-tile sort: shared-memory merge sort of the 64-bit local keys ------------------------------------------------
// One CTA per tile.  Each thread sorts 8 consecutive keys in registers (odd-even merge network, 19 compare-exchanges),
// then log2(n/8) merge passes ping-pong between two shared buffers; in a pass every thread produces 8 consecutive
// outputs: it locates its start in the two input runs with a merge-path binary search and merges sequentially.
// ~100 instructions per key in total (a shared-memory bitonic network needs ~500).
constexpr int SORT_VT = 8;
constexpr uint64_t KEY_MAX = 0xFFFFFFFFFFFFFFFFull;

__device__ __forceinline__ void cswap(uint64_t& a, uint64_t& b) {
	const uint64_t lo = a < b ? a : b, hi = a < b ? b : a;
	a = lo;
	b = hi;
}

// Shared-memory index with one pad slot per 16 keys: a thread's merge window starts ~4 keys after its neighbour's,
// i.e. 32 B apart -- unpadded that is an 8-way bank conflict on every step of the merge.
__device__ __forceinline__ int spad(int e) { return e + (e >> 4); }
constexpr int SORT_THREADS = 128;

// Sort `n` (<= the capacity the two buffers were sized for) 64-bit keys from global memory into shared memory; returns the
// buffer that holds the sorted run.  Runs of 8 straight from global memory through a register network (Batcher odd-even merge
// sort, 19 compare-exchanges), then merge-path passes ping-ponging between the two buffers.
__device__ __forceinline__ uint64_t* sort_in_shared(const uint64_t* __restrict__ src, int n, uint64_t* bufA, uint64_t* bufB) {
	const int tid = threadIdx.x, nthreads = blockDim.x;
	for (int o0 = tid * SORT_VT; o0 < n; o0 += nthreads * SORT_VT) {
		uint64_t k[SORT_VT];
#pragma unroll
		for (int q = 0; q < SORT_VT; q++) k[q] = (o0 + q < n) ? src[o0 + q] : KEY_MAX;
		cswap(k[0], k[1]); cswap(k[2], k[3]); cswap(k[4], k[5]); cswap(k[6], k[7]);
		cswap(k[0], k[2]); cswap(k[1], k[3]); cswap(k[4], k[6]); cswap(k[5], k[7]);
		cswap(k[1], k[2]); cswap(k[5], k[6]);
		cswap(k[0], k[4]); cswap(k[1], k[5]); cswap(k[2], k[6]); cswap(k[3], k[7]);
		cswap(k[2], k[4]); cswap(k[3], k[5]);
		cswap(k[1], k[2]); cswap(k[3], k[4]); cswap(k[5], k[6]);
#pragma unroll
		for (int q = 0; q < SORT_VT; q++)
			if (o0 + q < n) bufA[spad(o0 + q)] = k[q];
	}
	__syncthreads();
	uint64_t* in = bufA;
	uint64_t* out = bufB;
	for (int L = SORT_VT; L < n; L <<= 1) {
		for (int o0 = tid * SORT_VT; o0 < n; o0 += nthreads * SORT_VT) {
			const int base = (o0 / (2 * L)) * (2 * L);
			const int a0 = base, lenA = min(L, n - base);
			const int b0 = base + lenA, lenB = max(0, min(L, n - b0));
			const int diag = o0 - base;
			int lo = max(0, diag - lenB), hi = min(diag, lenA);
			while (lo < hi) {  // merge path: smallest i with A[i] > B[diag-1-i]
				const int mid = (lo + hi) >> 1;
				if (in[spad(a0 + mid)] <= in[spad(b0 + diag - 1 - mid)]) lo = mid + 1; else hi = mid;
			}
			int i = lo, j = diag - lo;
			uint64_t ka = i < lenA ? in[spad(a0 + i)] : KEY_MAX, kb = j < lenB ? in[spad(b0 + j)] : KEY_MAX;
#pragma unroll
			for (int q = 0; q < SORT_VT; q++) {
				if (o0 + q < n) {
					const bool take_a = ka <= kb;  // exhausted runs read as KEY_MAX; keys are unique, KEY_MAX never occurs
					out[spad(o0 + q)] = take_a ? ka : kb;
					if (take_a) { i++; ka = i < lenA ? in[spad(a0 + i)] : KEY_MAX; } else { j++; kb = j < lenB ? in[spad(b0 + j)] : KEY_MAX; }
				}
			}
		}
		__syncthreads();
		uint64_t* t = in; in = out; out = t;
	}
	return in;
}

__global__ void __launch_bounds__(SORT_THREADS) tile_sort_kernel(const uint2* __restrict__ ranges, int grid_x, int row_begin,
                                                                  const uint64_t* __restrict__ local_keys, uint32_t* __restrict__ point_list,
                                                                  uint64_t* __restrict__ keys_sorted, int cap) {
	extern __shared__ uint64_t s_keys[];  // [2][spad(cap)]
	const int tile = (blockIdx.y + row_begin) * grid_x + blockIdx.x;
	const uint2 rg = ranges[tile];
	const int n = (int)(rg.y - rg.x);
	if (n == 0 || n > cap) return;  // longer lists: the multi-CTA path below
	const int tid = threadIdx.x;
	const uint64_t* in = sort_in_shared(local_keys + rg.x, n, s_keys, s_keys + spad(cap));
	uint32_t* dst = point_list + rg.x;
	uint64_t* kdst = keys_sorted + rg.x;
	const uint64_t tile_hi = (uint64_t)tile << 32;
	for (int i = tid; i < n; i += SORT_THREADS) {
		const uint64_t k = in[spad(i)];
		dst[i] = (uint32_t)k;
		kdst[i] = tile_hi | (k >> 32);
	}
}

// ---- tile lists longer than the shared-memory capacity: split -> sort chunks -> merge, several CTAs per tile ---------------------
// Only the long tiles take this path; every other tile is finished by tile_sort_kernel above and is not touched here (the
// CTAs of short tiles leave at once).  Grid = (tiles of the slab) x (chunks of the longest list).
//   1. long_chunk_sort_kernel: CTA (tile, c) sorts elements [c*LONG_CHUNK, (c+1)*LONG_CHUNK) of the tile's segment in shared
//      memory and writes the sorted run back in place;
//   2. long_merge_kernel, run length L = LONG_CHUNK, 2*LONG_CHUNK, ...: CTA (tile, c) produces outputs [c*LONG_CHUNK, ...) of
//      the merge of the pair of runs they fall into: two merge-path searches in global memory bound the input ranges, those
//      LONG_CHUNK inputs are staged in shared memory, every thread merges LONG_VT consecutive outputs.  Ping-pong between the
//      local-key buffer and the (not yet written) exported-key buffer of the same segment;
//   3. long_finalize_kernel: local keys -> sorted ids + exported (tile | depth) keys.
// Equal depth bits order by Gaussian index through the low key half, as everywhere else (the reference's stable radix sort).
constexpr int LONG_CHUNK = 4096;
constexpr int LONG_THREADS = 256;
constexpr int LONG_VT = LONG_CHUNK / LONG_THREADS;

__global__ void __launch_bounds__(LONG_THREADS) long_chunk_sort_kernel(const uint2* __restrict__ ranges, int grid_x, int row_begin, int cap,
                                                                        uint64_t* __restrict__ local_keys) {
	extern __shared__ uint64_t s_keys[];  // [2][spad(LONG_CHUNK)]
	const int tile = (blockIdx.y + row_begin) * grid_x + blockIdx.x;
	const uint2 rg = ranges[tile];
	const int n = (int)(rg.y - rg.x);
	const int c0 = blockIdx.z * LONG_CHUNK;
	if (n <= cap || c0 >= n) return;
	const int m = min(LONG_CHUNK, n - c0);
	uint64_t* seg = local_keys + rg.x + c0;
	const uint64_t* in = sort_in_shared(seg, m, s_keys, s_keys + spad(LONG_CHUNK));  // reads all of `seg` before its first barrier
	for (int i = threadIdx.x; i < m; i += LONG_THREADS) seg[i] = in[spad(i)];
}

// smallest i in [max(0, d - lenB), min(d, lenA)] with A[i] > B[d - 1 - i]: the first d outputs of merge(A, B) take i from A
__device__ __forceinline__ int merge_path(const uint64_t* __restrict__ A, int lenA, const uint64_t* __restrict__ B, int lenB, int d) {
	int lo = max(0, d - lenB), hi = min(d, lenA);
	while (lo < hi) {
		const int mid = (lo + hi) >> 1;
		if (A[mid] <= B[d - 1 - mid]) lo = mid + 1; else hi = mid;
	}
	return lo;
}

__global__ void __launch_bounds__(LONG_THREADS) long_merge_kernel(const uint2* __restrict__ ranges, int grid_x, int row_begin, int cap, int L,
                                                                   const uint64_t* __restrict__ src, uint64_t* __restrict__ dst) {
	__shared__ uint64_t s_in[LONG_CHUNK];
	__shared__ int s_split[2];
	const int tile = (blockIdx.y + row_begin) * grid_x + blockIdx.x;
	const uint2 rg = ranges[tile];
	const int n = (int)(rg.y - rg.x);
	const int o0 = blockIdx.z * LONG_CHUNK;
	if (n <= cap || o0 >= n) return;
	const int o1 = min(n, o0 + LONG_CHUNK);
	const int tid = threadIdx.x;
	const int base = (o0 / (2 * L)) * (2 * L);
	const int lenA = min(L, n - base), lenB = max(0, min(L, n - base - lenA));
	const uint64_t* A = src + rg.x + base;
	const uint64_t* B = A + lenA;
	if (tid < 2) s_split[tid] = merge_path(A, lenA, B, lenB, (tid == 0 ? o0 : o1) - base);
	__syncthreads();
	const int a0 = s_split[0], a1 = s_split[1];
	const int b0 = (o0 - base) - a0, b1 = (o1 - base) - a1;
	const int na = a1 - a0, nb = b1 - b0;  // na + nb = o1 - o0 <= LONG_CHUNK
	for (int i = tid; i < na; i += LONG_THREADS) s_in[i] = A[a0 + i];
	for (int i = tid; i < nb; i += LONG_THREADS) s_in[na + i] = B[b0 + i];
	__syncthreads();
	const uint64_t* sA = s_in;
	const uint64_t* sB = s_in + na;
	const int total = na + nb;
	const int d0 = min(total, tid * LONG_VT);
	int i = merge_path(sA, na, sB, nb, d0), j = d0 - i;
	uint64_t ka = i < na ? sA[i] : KEY_MAX, kb = j < nb ? sB[j] : KEY_MAX;
	uint64_t* out = dst + rg.x + o0;
#pragma unroll 4
	for (int q = 0; q < LONG_VT; q++) {
		if (d0 + q < total) {
			const bool take_a = ka <= kb;
			out[d0 + q] = take_a ? ka : kb;
			if (take_a) { i++; ka = i < na ? sA[i] : KEY_MAX; } else { j++; kb = j < nb ? sB[j] : KEY_MAX; }
		}
	}
}

__global__ void __launch_bounds__(LONG_THREADS) long_finalize_kernel(const uint2* __restrict__ ranges, int grid_x, int row_begin, int cap,
                                                                      const uint64_t* src, uint32_t* __restrict__ point_list, uint64_t* keys_sorted) {
	const int tile = (blockIdx.y + row_begin) * grid_x + blockIdx.x;
	const uint2 rg = ranges[tile];
	const int n = (int)(rg.y - rg.x);
	const int o0 = blockIdx.z * LONG_CHUNK;
	if (n <= cap || o0 >= n) return;
	const int o1 = min(n, o0 + LONG_CHUNK);
	const uint64_t tile_hi = (uint64_t)tile << 32;
	for (int i = o0 + threadIdx.x; i < o1; i += LONG_THREADS) {
		const uint64_t k = src[rg.x + i];  // src may BE keys_sorted (odd number of merge passes): element-wise in place
		point_list[rg.x + i] = (uint32_t)k;
		keys_sorted[rg.x + i] = tile_hi | (k >> 32);
	}
}

void launch_tile_binning(const FwdParams& p, GeomView g, BinView b, ImgView img, const int* radii, int64_t R, uint32_t max_list, cudaStream_t s) {
	if (R <= 0 || p.row_end <= p.row_begin) return;
	scatter_kernel<<<(p.P + 255) / 256, 256, 0, s>>>(p.P, g.records, rec_floats(p.coord), g.depths, g.tiles_touched, radii, p.grid_x, p.grid_y,
	                                                  p.row_begin, p.row_end, img.ranges, img.tile_count, b.keys_unsorted);
	const int longest_short = (int)min(max_list, (uint32_t)TILE_SORT_CAP);
	const int cap = (max(longest_short, 256) + 255) & ~255;  // keys per ping-pong buffer
	const size_t smem = (size_t)2 * (cap + (cap >> 4)) * sizeof(uint64_t);
	static size_t configured[64] = {};
	if (smem > 48 * 1024) ensure_dynamic_smem(tile_sort_kernel, (size_t)2 * (TILE_SORT_CAP + (TILE_SORT_CAP >> 4)) * sizeof(uint64_t), configured);
	dim3 grid(p.grid_x, p.row_end - p.row_begin, 1);
	tile_sort_kernel<<<grid, SORT_THREADS, smem, s>>>(img.ranges, p.grid_x, p.row_begin, b.keys_unsorted, b.point_list, b.keys_sorted, cap);
	count_launch(2);
	if (max_list > (uint32_t)TILE_SORT_CAP) {
		const int chunks = (int)((max_list + LONG_CHUNK - 1) / LONG_CHUNK);
		dim3 lgrid(p.grid_x, p.row_end - p.row_begin, chunks);
		const size_t lsmem = (size_t)2 * (LONG_CHUNK + (LONG_CHUNK >> 4)) * sizeof(uint64_t);
		static size_t lconfigured[64] = {};
		ensure_dynamic_smem(long_chunk_sort_kernel, lsmem, lconfigured);
		long_chunk_sort_kernel<<<lgrid, LONG_THREADS, lsmem, s>>>(img.ranges, p.grid_x, p.row_begin, TILE_SORT_CAP, b.keys_unsorted);
		uint64_t* src = b.keys_unsorted;
		uint64_t* dst = b.keys_sorted;
		int launches = 2;
		for (int64_t L = LONG_CHUNK; L < (int64_t)max_list; L <<= 1) {
			long_merge_kernel<<<lgrid, LONG_THREADS, 0, s>>>(img.ranges, p.grid_x, p.row_begin, TILE_SORT_CAP, (int)L, src, dst);
			uint64_t* t = src; src = dst; dst = t;
			launches++;
		}
		long_finalize_kernel<<<lgrid, LONG_THREADS, 0, s>>>(img.ranges, p.grid_x, p.row_begin, TILE_SORT_CAP, src, b.point_list, b.keys_sorted);
		count_launch(launches);
	}
}

}  // namespace rgs
