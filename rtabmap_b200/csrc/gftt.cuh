// gftt.cuh — GFTT corners for Kp/DetectorStrategy=8 (GFTT/ORB, RTAB-Map's default detector): the DETECT half.
//
// Replaces: GFTT::generateKeypointsImpl (corelib/src/Features2d.cpp:2148-2178), i.e. OpenCV's cv::GFTTDetector::detect =
// goodFeaturesToTrack with the min-eigenvalue score (cornerMinEigenVal, blockSize, Sobel aperture 3).  The descriptors
// (GFTT_ORB::generateDescriptorsImpl, :2351-2355 -> cv::ORB::compute with the provided keypoints) reuse orb.cuh's level-0
// blur, steered BRIEF and 3-D lifting unchanged.  oracle/gftt_py.py is the written spec of the arithmetic below and
// tests/test_oracle_gftt.py pins it to opencv-python 4.13:
//   * Sobel, scale = 1 / (4 * blockSize * 255), k0 = float(scale), k1 = float(2 * scale), BORDER_REFLECT_101:
//     dx = fmaf(r[y-1] + r[y+1], k0, r[y] * k1) over the exact integer row differences r = p[x+1] - p[x-1];
//     dy = R[y+1] - R[y-1] over R = fmaf(p[x+1], k0, fmaf(p[x], k1, p[x-1] * k0)), except in the columns past the last
//     multiple of 16 (the scalar tail of OpenCV's vector loop): R = (p[x-1] * k0 + p[x] * k1) + p[x+1] * k0;
//   * dx*dx, dx*dy, dy*dy in float; unnormalised box filter: row sums in double (direct, left to right, for 3 and 5 taps;
//     a running s += new - old along the whole row for 7), column sums a running double down the whole frame
//     (s = SUM + new; out = float(s); SUM = s - old);
//   * lambda = (a + c) - sqrtf((a - c)^2 + b^2), a = cxx * 0.5f, c = cyy * 0.5f, no FMA (the build uses --fmad=false; the
//     fused operations above are explicit __fmaf_rn);
//   * selection: THRESH_TOZERO at float(maxVal * qualityLevel) (maxVal over the mask), 3x3 local maximum, interior
//     [1, h-2] x [1, w-2], mask; order lambda descending then address descending; greedy min-distance pass over a grid of
//     cvRound(minDistance) cells (+-1 cell, rejected when dx^2 + dy^2 < minDistance^2), maxCorners.
#pragma once
#include "common.cuh"
#include "orb.cuh"
#include <assert.h>

namespace lcd {

constexpr int kGfttCandCap = 65536;      // candidates (local maxima above the quality threshold) kept per frame
constexpr int kGfttSelectThreads = 1024;
constexpr int kGfttSortCap = 8192;       // keys sorted in shared memory at a time (64 KB); larger lists go chunk by chunk
// Accepted corners per grid cell: a cell has side c = cvRound(d) <= d + 1/2 (d = minDistance >= 1); split into four
// sub-squares of ceil(c/2) pixels, two pixels of one sub-square lie at most sqrt(2) * (c - 1) / 2 <= 0.71 (d - 1/2) < d
// apart, so each sub-square holds at most one accepted corner.  The occupancy bitmap below needs no per-cell storage;
// the bound is what keeps the per-candidate window scan short (at most 9 cells x 4 corners), and the selection kernel asserts it.
constexpr int kGfttCellMax = 4;
static_assert(kGfttSortCap % 32 == 0, "the greedy pass walks the sorted chunk in warps of 32");

// ordered bits: the unsigned order of the result is the float order (negative values included)
__device__ __forceinline__ uint32_t f32_ordered(float f)
{
	const uint32_t u = __float_as_uint(f);
	return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float f32_from_ordered(uint32_t k)
{
	return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}

struct GfttArgs
{
	const uint8_t * gray; // level 0 of the ORB workspace: [n_frames][frame_stride]
	const uint8_t * mask; // same layout, or nullptr
	int w, h, frame_stride;
	float k0, k1;         // Sobel coefficients (scale, 2 * scale)
	float * eig;          // [n_frames][h][w] minimum eigenvalue
	uint32_t * max_bits;  // [n_frames] ordered bits of the largest eigenvalue inside the mask (0: none yet)
	double * rowsum;      // blockSize 7 only: [n_frames][h][w][3] row sums of the products
};

// Sobel dx, dy at (x, y) in OpenCV's operation order, and the three products
__device__ __forceinline__ void gftt_products(const uint8_t * img, int w, int h, int x, int y, float k0, float k1, float & pxx, float & pxy, float & pyy)
{
	const int xm = reflect101(x - 1, w), xp = reflect101(x + 1, w);
	const int rows[3] = {reflect101(y - 1, h), y, reflect101(y + 1, h)};
	const bool tail = x >= (w & ~15);
	float rx[3], ry[3];
#pragma unroll
	for (int i = 0; i < 3; ++i)
	{
		const uint8_t * r = img + static_cast<size_t>(rows[i]) * w;
		const int L = r[xm], C = r[x], R = r[xp];
		rx[i] = static_cast<float>(R - L);
		const float Lf = static_cast<float>(L), Cf = static_cast<float>(C), Rf = static_cast<float>(R);
		ry[i] = tail ? __fadd_rn(__fadd_rn(__fmul_rn(Lf, k0), __fmul_rn(Cf, k1)), __fmul_rn(Rf, k0))
		             : __fmaf_rn(Rf, k0, __fmaf_rn(Cf, k1, __fmul_rn(Lf, k0)));
	}
	const float dx = __fmaf_rn(__fadd_rn(rx[0], rx[2]), k0, __fmul_rn(rx[1], k1));
	const float dy = __fsub_rn(ry[2], ry[0]);
	pxx = __fmul_rn(dx, dx);
	pxy = __fmul_rn(dx, dy);
	pyy = __fmul_rn(dy, dy);
}

__device__ __forceinline__ float gftt_lambda(float cxx, float cxy, float cyy)
{
	const float a = __fmul_rn(cxx, 0.5f), c = __fmul_rn(cyy, 0.5f);
	const float t = __fsub_rn(a, c);
	return __fsub_rn(__fadd_rn(a, c), __fsqrt_rn(__fadd_rn(__fmul_rn(t, t), __fmul_rn(cxy, cxy))));
}

// The column pass shared by both eigenvalue kernels: B = blockSize row sums in a shift register, the running double sum,
// lambda, the masked maximum.  `next(t, s)` returns the row sums of extended row t (image row reflect101(t - R)).
template <int B, class Next>
__device__ __forceinline__ void gftt_column(const GfttArgs & a, int frame, int x, bool out, Next next)
{
	constexpr int R = B / 2;
	const int w = a.w, h = a.h;
	const uint8_t * mask = a.mask ? a.mask + static_cast<size_t>(frame) * a.frame_stride : nullptr;
	float * eig = a.eig + static_cast<size_t>(frame) * w * h;
	double hist[B - 1][3];
	double sum[3] = {0.0, 0.0, 0.0};
	uint32_t best = 0u;
	for (int t = 0; t < h + 2 * R; ++t)
	{
		double s[3];
		next(t, s);
		if (t < B - 1)
		{
#pragma unroll
			for (int c = 0; c < 3; ++c) sum[c] = sum[c] + s[c];
		}
		else
		{
			float o[3];
#pragma unroll
			for (int c = 0; c < 3; ++c)
			{
				const double v = sum[c] + s[c];
				o[c] = static_cast<float>(v);
				sum[c] = v - hist[0][c];
			}
			const int y = t - (B - 1);
			if (out)
			{
				const float lam = gftt_lambda(o[0], o[1], o[2]);
				eig[static_cast<size_t>(y) * w + x] = lam;
				if (!mask || mask[static_cast<size_t>(y) * w + x]) best = max(best, f32_ordered(lam));
			}
		}
#pragma unroll
		for (int k = 0; k < B - 2; ++k)
#pragma unroll
			for (int c = 0; c < 3; ++c) hist[k][c] = hist[k + 1][c];
#pragma unroll
		for (int c = 0; c < 3; ++c) hist[B - 2][c] = s[c];
	}
	best = __reduce_max_sync(0xFFFFFFFFu, best);
	if ((threadIdx.x & 31) == 0 && best) atomicMax(a.max_bits + frame, best);
}

// ---- G1: eigenvalue stencil, blockSize 3 and 5.  One warp per strip of 32 - 2R output columns: every lane computes the
// products of one column (the strip plus an R-column halo each side, reflected at the image border), the row sums come
// from shuffles, and each output lane carries its running double column sum down the whole frame.
template <int B>
__global__ void __launch_bounds__(128) gftt_eigen_kernel(const GfttArgs a)
{
	constexpr int R = B / 2, OW = 32 - 2 * R;
	const int lane = threadIdx.x & 31;
	const int strip = blockIdx.x * 4 + (threadIdx.x >> 5);
	const int frame = blockIdx.y;
	const int w = a.w, h = a.h;
	if (strip * OW >= w) return; // uniform per warp
	const int xo = strip * OW + lane - R;
	const int xc = reflect101(min(xo, w - 1 + R), w);
	const bool out = lane >= R && lane < 32 - R && xo < w;
	const uint8_t * img = a.gray + static_cast<size_t>(frame) * a.frame_stride;
	gftt_column<B>(a, frame, xo, out, [&](int t, double * s) {
		float p[3];
		gftt_products(img, w, h, xc, reflect101(t - R, h), a.k0, a.k1, p[0], p[1], p[2]);
#pragma unroll
		for (int c = 0; c < 3; ++c)
		{
			double v = static_cast<double>(__shfl_sync(0xFFFFFFFFu, p[c], (lane - R) & 31));
#pragma unroll
			for (int d = 1 - R; d <= R; ++d) v = v + static_cast<double>(__shfl_sync(0xFFFFFFFFu, p[c], (lane + d) & 31));
			s[c] = v;
		}
	});
}

// ---- G1 (blockSize 7): OpenCV's 7-tap row sum is a running sum along the whole row, so the rows go first (one thread
// per frame row, a sliding window of 7 products), the column pass second, one thread per column.
__global__ void __launch_bounds__(128) gftt_rowsum7_kernel(const GfttArgs a)
{
	const int y = blockIdx.x * blockDim.x + threadIdx.x;
	const int frame = blockIdx.y;
	const int w = a.w, h = a.h;
	if (y >= h) return;
	const uint8_t * img = a.gray + static_cast<size_t>(frame) * a.frame_stride;
	double * out = a.rowsum + (static_cast<size_t>(frame) * h + y) * w * 3;
	float win[7][3];
#pragma unroll
	for (int k = 0; k < 7; ++k) gftt_products(img, w, h, reflect101(k - 3, w), y, a.k0, a.k1, win[k][0], win[k][1], win[k][2]);
	double s[3];
#pragma unroll
	for (int c = 0; c < 3; ++c)
	{
		s[c] = static_cast<double>(win[0][c]);
#pragma unroll
		for (int k = 1; k < 7; ++k) s[c] = s[c] + static_cast<double>(win[k][c]);
		out[c] = s[c];
	}
	for (int x = 1; x < w; ++x)
	{
		float n[3];
		gftt_products(img, w, h, reflect101(x + 3, w), y, a.k0, a.k1, n[0], n[1], n[2]);
#pragma unroll
		for (int c = 0; c < 3; ++c)
		{
			s[c] = s[c] + (static_cast<double>(n[c]) - static_cast<double>(win[0][c]));
			out[static_cast<size_t>(x) * 3 + c] = s[c];
		}
#pragma unroll
		for (int k = 0; k < 6; ++k)
#pragma unroll
			for (int c = 0; c < 3; ++c) win[k][c] = win[k + 1][c];
#pragma unroll
		for (int c = 0; c < 3; ++c) win[6][c] = n[c];
	}
}

__global__ void __launch_bounds__(128) gftt_colsum7_kernel(const GfttArgs a)
{
	const int x = blockIdx.x * blockDim.x + threadIdx.x;
	const int frame = blockIdx.y;
	const int w = a.w, h = a.h;
	const bool out = x < w;
	const double * rs = a.rowsum + static_cast<size_t>(frame) * h * w * 3;
	const int xs = out ? x : w - 1;
	gftt_column<7>(a, frame, xs, out, [&](int t, double * s) {
		const double * r = rs + (static_cast<size_t>(reflect101(t - 3, h)) * w + xs) * 3;
		s[0] = r[0];
		s[1] = r[1];
		s[2] = r[2];
	});
}

// ---- G2: candidates.  THRESH_TOZERO, 3x3 local maximum of the thresholded map (the dilate), interior and mask test;
// keys (ordered lambda << 24 | address) appended to the frame's list, one atomic per warp.
__global__ void __launch_bounds__(256) gftt_candidate_kernel(const GfttArgs a, double quality_level, unsigned long long * __restrict__ cand,
                                                             int * __restrict__ cand_count, int * __restrict__ overflow)
{
	const int x = blockIdx.x * blockDim.x + threadIdx.x;
	const int y = blockIdx.y * blockDim.y + threadIdx.y;
	const int frame = blockIdx.z;
	const int w = a.w, h = a.h;
	const int lane = (threadIdx.y * blockDim.x + threadIdx.x) & 31;
	const uint32_t mb = a.max_bits[frame];
	const double max_val = mb ? static_cast<double>(f32_from_ordered(mb)) : 0.0;
	const float thr = static_cast<float>(max_val * quality_level);
	const float * eig = a.eig + static_cast<size_t>(frame) * w * h;
	bool keep = false;
	float v = 0.f;
	if (x >= 1 && x < w - 1 && y >= 1 && y < h - 1)
	{
		v = eig[static_cast<size_t>(y) * w + x];
		if (v > thr)
		{
			keep = true;
#pragma unroll
			for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
				for (int dx = -1; dx <= 1; ++dx)
				{
					const float n = eig[static_cast<size_t>(y + dy) * w + x + dx];
					if (n > thr && n > v) keep = false;
				}
			if (keep && a.mask && a.mask[static_cast<size_t>(frame) * a.frame_stride + static_cast<size_t>(y) * w + x] == 0) keep = false;
		}
	}
	const unsigned m = __ballot_sync(0xFFFFFFFFu, keep);
	if (!m) return;
	int base = 0;
	if (lane == 0) base = atomicAdd(&cand_count[frame], __popc(m));
	base = __shfl_sync(0xFFFFFFFFu, base, 0);
	if (keep)
	{
		const int k = base + __popc(m & ((1u << lane) - 1u));
		if (k < kGfttCandCap)
			cand[static_cast<size_t>(frame) * kGfttCandCap + k] = (static_cast<unsigned long long>(f32_ordered(v)) << 24) | static_cast<unsigned>(y * w + x);
		else atomicExch(overflow, 1);
	}
}

// ---- G3: selection, one CTA per frame ---------------------------------------------------------------------------------
struct GfttSelectArgs
{
	const unsigned long long * cand;
	const int * cand_count;
	int w, h;
	double min_distance, min_distance2;
	int cell;          // cvRound(minDistance); 0: no distance test (minDistance < 1)
	int max_corners;
	int edge;          // ORB/EdgeThreshold: ORB::compute's KeyPointsFilter::runByImageBorder
	int block_size;
	uint32_t * occ_global; // [n_frames][h][ceil(w/32)] occupancy bitmap when it does not fit in shared memory, else nullptr
	OrbKeypoint * kp;  // [n_frames][cap]
	int * n_kp;        // [n_frames]
	int cap;
};

__device__ __forceinline__ uint32_t gftt_occ_load(const uint32_t * occ, bool global, int i)
{
	return global ? __ldcg(occ + i) : occ[i];
}

__global__ void __launch_bounds__(kGfttSelectThreads) gftt_select_kernel(const GfttSelectArgs a)
{
	extern __shared__ __align__(16) unsigned char smem_raw[];
	unsigned long long * s_keys = reinterpret_cast<unsigned long long *>(smem_raw); // [kGfttSortCap]
	__shared__ int s_hist[256];
	__shared__ unsigned long long s_prefix;
	__shared__ int s_need, s_m, s_done;
	const int tid = threadIdx.x, lane = tid & 31;
	const int frame = blockIdx.x;
	const int w = a.w, h = a.h, wpr = (w + 31) >> 5;
	const bool occ_in_global = a.occ_global != nullptr;
	uint32_t * occ = occ_in_global ? a.occ_global + static_cast<size_t>(frame) * h * wpr : reinterpret_cast<uint32_t *>(s_keys + kGfttSortCap);
	const unsigned long long * keys = a.cand + static_cast<size_t>(frame) * kGfttCandCap;
	const int n = min(a.cand_count[frame], kGfttCandCap);
	if (a.cell > 0)
		for (int i = tid; i < h * wpr; i += blockDim.x) occ[i] = 0u;
	if (tid == 0) s_done = 0;
	__syncthreads();
	// warp 0's running state (registers, uniform across the warp)
	int accepted = 0, n_out = 0;
	unsigned long long upper = ~0ull; // the next chunk holds the largest keys below `upper`
	int consumed = 0;
	while (consumed < n)
	{
		const int rem = n - consumed;
		unsigned long long lo = 0ull;
		if (rem > kGfttSortCap)
		{
			// radix select (8-bit digits, 56-bit keys): lo = the kGfttSortCap-th largest key below `upper`
			if (tid == 0)
			{
				s_prefix = 0ull;
				s_need = kGfttSortCap;
			}
			for (int shift = 48; shift >= 0; shift -= 8)
			{
				for (int i = tid; i < 256; i += blockDim.x) s_hist[i] = 0;
				__syncthreads();
				const unsigned long long pre = s_prefix;
				for (int i = tid; i < n; i += blockDim.x)
				{
					const unsigned long long k = keys[i];
					if (k < upper && (k >> (shift + 8)) == (pre >> (shift + 8))) atomicAdd(&s_hist[(k >> shift) & 255], 1);
				}
				__syncthreads();
				if (tid == 0)
				{
					int need = s_need, cum = 0, b = 255;
					for (; b > 0; --b)
					{
						if (cum + s_hist[b] >= need) break;
						cum += s_hist[b];
					}
					s_need = need - cum;
					s_prefix = pre | (static_cast<unsigned long long>(b) << shift);
				}
				__syncthreads();
			}
			lo = s_prefix;
		}
		// gather the chunk [lo, upper) and sort it, descending (bitonic, zero padding sorts last)
		if (tid == 0) s_m = 0;
		__syncthreads();
		for (int i = tid; i < n; i += blockDim.x)
		{
			const unsigned long long k = keys[i];
			if (k >= lo && k < upper) s_keys[atomicAdd(&s_m, 1)] = k;
		}
		__syncthreads();
		const int m = s_m;
		int pad = 32;
		while (pad < m) pad <<= 1;
		for (int i = m + tid; i < pad; i += blockDim.x) s_keys[i] = 0ull;
		__syncthreads();
		for (int k = 2; k <= pad; k <<= 1)
			for (int j = k >> 1; j > 0; j >>= 1)
			{
				for (int i = tid; i < pad; i += blockDim.x)
				{
					const int ixj = i ^ j;
					if (ixj > i)
					{
						const unsigned long long x = s_keys[i], y = s_keys[ixj];
						if ((x < y) == ((i & k) == 0))
						{
							s_keys[i] = y;
							s_keys[ixj] = x;
						}
					}
				}
				__syncthreads();
			}
		// greedy min-distance pass, warp 0, 32 candidates at a time.  A candidate is rejected by the corners accepted in
		// earlier groups (occupancy bitmap) or by an accepted earlier candidate of its own group; the latter is settled by a
		// ballot fixed point: each round accepts the undecided lanes with no undecided or accepted earlier conflict and
		// rejects those with an accepted one, so the lowest undecided lane is always decided and the result is the
		// sequential one.
		if (tid < 32)
		{
			for (int base = 0; base < m; base += 32)
			{
				const int j = base + lane;
				const bool valid = j < m;
				const unsigned long long key = valid ? s_keys[j] : 0ull;
				const int idx = static_cast<int>(key & 0xFFFFFFull);
				const int x = idx % w, y = idx / w;
				unsigned A;
				if (a.cell > 0)
				{
					const int c = a.cell, xc = x / c, yc = y / c;
					bool alive = valid;
					if (alive)
					{
						const int x0 = max(xc - 1, 0) * c, x1 = min((xc + 2) * c, w) - 1;
						const int y0 = max(yc - 1, 0) * c, y1 = min((yc + 2) * c, h) - 1;
						int seen = 0;
						for (int yy = y0; yy <= y1 && alive; ++yy)
							for (int wd = x0 >> 5; wd <= (x1 >> 5) && alive; ++wd)
							{
								uint32_t bits = gftt_occ_load(occ, occ_in_global, yy * wpr + wd);
								if (wd == (x0 >> 5)) bits &= ~0u << (x0 & 31);
								if (wd == (x1 >> 5) && (x1 & 31) != 31) bits &= (2u << (x1 & 31)) - 1u;
								for (; bits; bits &= bits - 1u)
								{
									const int px = wd * 32 + __ffs(bits) - 1;
									const double d2 = static_cast<double>((px - x) * (px - x) + (yy - y) * (yy - y));
									++seen;
									if (d2 < a.min_distance2)
									{
										alive = false;
										break;
									}
								}
							}
						assert(seen <= 9 * kGfttCellMax);
					}
					unsigned cm = 0u; // earlier lanes of this group that would reject this one
#pragma unroll 4
					for (int i = 0; i < 32; ++i)
					{
						const int xi = __shfl_sync(0xFFFFFFFFu, x, i), yi = __shfl_sync(0xFFFFFFFFu, y, i);
						const int dxc = xi / c - xc, dyc = yi / c - yc;
						const double d2 = static_cast<double>((xi - x) * (xi - x) + (yi - y) * (yi - y));
						if (i < lane && dxc >= -1 && dxc <= 1 && dyc >= -1 && dyc <= 1 && d2 < a.min_distance2) cm |= 1u << i;
					}
					unsigned U = __ballot_sync(0xFFFFFFFFu, alive);
					A = 0u;
					while (U)
					{
						const bool mine = (U >> lane) & 1u;
						const unsigned acc = __ballot_sync(0xFFFFFFFFu, mine && (cm & (U | A)) == 0u);
						const unsigned rej = __ballot_sync(0xFFFFFFFFu, mine && (cm & A) != 0u);
						A |= acc;
						U &= ~(acc | rej);
					}
				}
				else A = __ballot_sync(0xFFFFFFFFu, valid);
				// maxCorners: the first `room` accepted corners of the group, in order
				const int room = a.max_corners - accepted;
				bool stop = false;
				if (__popc(A) >= room)
				{
					unsigned t = A;
					for (int r = 0; r < room; ++r) t &= t - 1u;
					A &= ~t;
					stop = true;
				}
				accepted += __popc(A);
				const bool mine = (A >> lane) & 1u;
				if (a.cell > 0 && mine) atomicOr(occ + y * wpr + (x >> 5), 1u << (x & 31));
				// ORB::compute drops the corners within ORB/EdgeThreshold of the border, keeping the order
				const bool keep = mine && x >= a.edge && x < w - a.edge && y >= a.edge && y < h - a.edge;
				const unsigned km = __ballot_sync(0xFFFFFFFFu, keep);
				const int pos = n_out + __popc(km & ((1u << lane) - 1u));
				if (keep && pos < a.cap)
				{
					OrbKeypoint kp;
					kp.x = static_cast<float>(x);
					kp.y = static_cast<float>(y);
					kp.size = static_cast<float>(a.block_size);
					kp.angle = -1.f;
					kp.response = f32_from_ordered(static_cast<uint32_t>(key >> 24));
					kp.octave = 0;
					a.kp[static_cast<size_t>(frame) * a.cap + pos] = kp;
				}
				n_out += __popc(km);
				__syncwarp();
				if (stop) break;
			}
			if (lane == 0 && accepted >= a.max_corners) s_done = 1;
		}
		__syncthreads();
		consumed += m;
		upper = lo;
		if (s_done || m == 0) break;
	}
	if (tid == 0) a.n_kp[frame] = min(n_out, a.cap);
}

} // namespace lcd
