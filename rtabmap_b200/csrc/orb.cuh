// orb.cuh — ORB keypoint detection and description on the incoming frame (the DETECT stage).
//
// Replaces: Feature2D::generateKeypoints / generateDescriptors / generateKeypoints3D for
// Kp/DetectorStrategy=2 (corelib/src/Features2d.cpp:775-878, :1621-1718, :905-1116), i.e. OpenCV's
// cv::ORB::detect + compute [third-party; algorithm restated in-tree at corelib/src/opencv/Orb.cpp:61-134
// (Harris, IC angle), :138-258 (steered BRIEF), :737-852 (pyramid + FAST + retainBest)], the depth mask
// (Features2d.cpp:783-808), Feature2D::limitKeypoints (:356-399), cv::cvtColor(BGR2GRAY) (Memory.cpp:5447)
// and util3d::generateKeypoints3DDepth (util3d_features.cpp:67-120; util2d::getDepth, util2d.cpp:947-1108).
//
// Bit-exactness notes (each pinned against opencv-python 4.13, tests/test_gpu_orb.py):
//   * gray = (B*3735 + G*19235 + R*9798 + 2^14) >> 15;
//   * pyramid (ORB/ScaleFactor = 2 only): INTER_LINEAR_EXACT by exactly 2 = (a+b+c+d+2) >> 2, level l from
//     level l-1; mask levels = 2x2 AND (resize + THRESH_TOZERO 254);
//   * FAST-9/16 score = max over the 16 arcs of the min |difference| - 1, 3x3 strict non-max suppression,
//     keypoints in raster order; border (ORB/EdgeThreshold) and mask filters after suppression;
//   * KeyPointsFilter::retainBest keeps ties and leaves the keypoints in the order libstdc++'s
//     std::nth_element (introselect, median-of-3, unguarded Hoare partition) and std::partition produce;
//     that order is the order of the frame's descriptors and therefore of its words, so the two
//     algorithms are replayed literally (sequentially, one thread per frame and level);
//   * Harris response and IC angle use float arithmetic in OpenCV's operation order, without FMA;
//     fastAtan2's polynomial coefficients are float products (c * 57.29578f);
//   * the 7x7 sigma=2 blur runs on a sub-matrix of the pyramid buffer, which sends OpenCV down the float
//     sepFilter2D path (not the fixed-point one): row pass in plain order, column pass symmetric, both with
//     fused multiply-add (AVX2 dispatch), round-to-nearest-even to uint8; descriptor taps that fall outside
//     the level read the UNBLURRED reflected border.
#pragma once
#include "common.cuh"
#include "orb_pattern.h"
#include <math.h>

namespace lcd {

constexpr int kOrbMaxLevels = 4;
constexpr int kOrbCandCap = 16384; // FAST corners kept per frame and level before retainBest
constexpr int kOrbSelectThreads = 512;
static_assert(kOrbCandCap <= 32 * kOrbSelectThreads, "partition_replay keeps one 32-bit stop mask per thread");

struct OrbKeypoint // cv::KeyPoint fields used by the reference
{
	float x, y, size, angle, response;
	int octave;
};

struct OrbGeom
{
	int n_levels;
	int w[kOrbMaxLevels], h[kOrbMaxLevels];
	int off[kOrbMaxLevels]; // plane offset of each level inside one frame's pyramid
	int frame_stride;       // bytes of one frame's pyramid
	int n_per_level[kOrbMaxLevels];
	int edge, fast_thr, patch;
};

__device__ __forceinline__ int reflect101(int i, int n)
{
	if (i < 0) i = -i;
	if (i >= n) i = 2 * n - 2 - i;
	return i;
}

// ---- K1: gray + depth mask (level 0) and level 1 -------------------------------------------------
// One thread per level-1 pixel (a 2x2 block of the input).
struct OrbPrepArgs
{
	const uint8_t * images; // [n_frames][h][w][channels]
	int channels;
	const void * depth;     // [n_frames][h][w] u16 (mm) or f32 (m), or nullptr
	int depth_type;         // 0 none, 1 u16, 2 f32, 3 u8 mask
	float min_depth, max_depth;
	uint8_t * gray;         // pyramids
	uint8_t * mask;         // pyramids or nullptr
	OrbGeom g;
};

__device__ __forceinline__ uint8_t depth_to_mask(const void * depth, int type, size_t idx, float min_depth, float max_depth)
{
	float value = 0.0f;
	if (type == 3) return static_cast<const uint8_t *>(depth)[idx] ? 255 : 0; // a ready-made CV_8UC1 mask (0 / 255)
	if (type == 1)
	{
		const unsigned short d = static_cast<const unsigned short *>(depth)[idx];
		if (d > 0 && d < 65535) value = static_cast<float>(d) * 0.001f;
	}
	else
	{
		value = static_cast<const float *>(depth)[idx];
	}
	return (value > min_depth && (max_depth == 0.0f || value <= max_depth) && isfinite(value)) ? 255 : 0;
}

__global__ void orb_prepare_kernel(const OrbPrepArgs a)
{
	const int x1 = blockIdx.x * blockDim.x + threadIdx.x;
	const int y1 = blockIdx.y * blockDim.y + threadIdx.y;
	const int frame = blockIdx.z;
	const int w = a.g.w[0], h = a.g.h[0];
	if (x1 * 2 >= w || y1 * 2 >= h) return;
	uint8_t * gray = a.gray + static_cast<size_t>(frame) * a.g.frame_stride;
	uint8_t * mask = a.mask ? a.mask + static_cast<size_t>(frame) * a.g.frame_stride : nullptr;
	const uint8_t * img = a.images + static_cast<size_t>(frame) * w * h * a.channels;
	int sum = 0;
	int mall = 255;
#pragma unroll
	for (int dy = 0; dy < 2; ++dy)
#pragma unroll
		for (int dx = 0; dx < 2; ++dx)
		{
			const int x = 2 * x1 + dx, y = 2 * y1 + dy;
			if (x >= w || y >= h) continue; // odd sizes (one pyramid level only)
			int gv;
			if (a.channels == 1) gv = img[static_cast<size_t>(y) * w + x];
			else
			{
				const uint8_t * p = img + (static_cast<size_t>(y) * w + x) * a.channels;
				gv = (p[0] * 3735 + p[1] * 19235 + p[2] * 9798 + (1 << 14)) >> 15;
			}
			gray[static_cast<size_t>(y) * w + x] = static_cast<uint8_t>(gv);
			sum += gv;
			if (mask)
			{
				const uint8_t m = depth_to_mask(a.depth, a.depth_type, static_cast<size_t>(frame) * w * h + static_cast<size_t>(y) * w + x, a.min_depth, a.max_depth);
				mask[static_cast<size_t>(y) * w + x] = m;
				mall &= m;
			}
		}
	if (a.g.n_levels > 1)
	{
		gray[a.g.off[1] + static_cast<size_t>(y1) * a.g.w[1] + x1] = static_cast<uint8_t>((sum + 2) >> 2);
		if (mask) mask[a.g.off[1] + static_cast<size_t>(y1) * a.g.w[1] + x1] = static_cast<uint8_t>(mall);
	}
}

// The same stage with 8 pixels x 2 rows per thread and vector loads / stores (rows that are a multiple of 8 pixels, even height, 16-byte
// aligned planes): ~1.5 instead of ~6.5 memory instructions per pixel.  Same integer arithmetic, same bytes out.
__global__ void __launch_bounds__(256)
orb_prepare_vec_kernel(const OrbPrepArgs a)
{
	const int xg = blockIdx.x * blockDim.x + threadIdx.x; // group of 8 level-0 pixels
	const int y1 = blockIdx.y * blockDim.y + threadIdx.y; // level-1 row
	const int frame = blockIdx.z;
	const int w = a.g.w[0], h = a.g.h[0];
	if (xg * 8 >= w || y1 * 2 >= h) return;
	uint8_t * gray = a.gray + static_cast<size_t>(frame) * a.g.frame_stride;
	uint8_t * mask = a.mask ? a.mask + static_cast<size_t>(frame) * a.g.frame_stride : nullptr;
	const size_t px = static_cast<size_t>(w) * h;
	const uint8_t * img = a.images + static_cast<size_t>(frame) * px * a.channels;
	int sum[4] = {0, 0, 0, 0};
	uint32_t mall = 0xFFFFFFFFu; // one byte per level-1 pixel
#pragma unroll
	for (int dy = 0; dy < 2; ++dy)
	{
		const int y = 2 * y1 + dy;
		const size_t at = static_cast<size_t>(y) * w + 8 * xg;
		int gv[8];
		if (a.channels == 1)
		{
			const uint2 v = *reinterpret_cast<const uint2 *>(img + at);
#pragma unroll
			for (int i = 0; i < 4; ++i)
			{
				gv[i] = (v.x >> (8 * i)) & 0xFF;
				gv[4 + i] = (v.y >> (8 * i)) & 0xFF;
			}
		}
		else
		{
			const uint2 * p = reinterpret_cast<const uint2 *>(img + at * 3);
			const uint2 q0 = p[0], q1 = p[1], q2 = p[2];
			const uint32_t wd[6] = {q0.x, q0.y, q1.x, q1.y, q2.x, q2.y};
#pragma unroll
			for (int i = 0; i < 8; ++i)
			{
				const int b0 = 3 * i, b1 = 3 * i + 1, b2 = 3 * i + 2;
				const int c0 = (wd[b0 >> 2] >> (8 * (b0 & 3))) & 0xFF, c1 = (wd[b1 >> 2] >> (8 * (b1 & 3))) & 0xFF, c2 = (wd[b2 >> 2] >> (8 * (b2 & 3))) & 0xFF;
				gv[i] = (c0 * 3735 + c1 * 19235 + c2 * 9798 + (1 << 14)) >> 15;
			}
		}
		uint2 gout;
		gout.x = gv[0] | (gv[1] << 8) | (gv[2] << 16) | (gv[3] << 24);
		gout.y = gv[4] | (gv[5] << 8) | (gv[6] << 16) | (gv[7] << 24);
		*reinterpret_cast<uint2 *>(gray + at) = gout;
#pragma unroll
		for (int i = 0; i < 8; ++i) sum[i >> 1] += gv[i];
		if (mask)
		{
			uint32_t m[8];
			const size_t di = static_cast<size_t>(frame) * px + at;
			if (a.depth_type == 3)
			{
				const uint2 v = *reinterpret_cast<const uint2 *>(static_cast<const uint8_t *>(a.depth) + di);
#pragma unroll
				for (int i = 0; i < 4; ++i)
				{
					m[i] = ((v.x >> (8 * i)) & 0xFF) ? 255u : 0u;
					m[4 + i] = ((v.y >> (8 * i)) & 0xFF) ? 255u : 0u;
				}
			}
			else
			{
				float val[8];
				if (a.depth_type == 1)
				{
					const uint4 v = *reinterpret_cast<const uint4 *>(static_cast<const unsigned short *>(a.depth) + di);
					const uint32_t dw[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
					for (int i = 0; i < 8; ++i)
					{
						const uint32_t d = (dw[i >> 1] >> (16 * (i & 1))) & 0xFFFFu;
						val[i] = (d > 0 && d < 65535) ? static_cast<float>(d) * 0.001f : 0.0f;
					}
				}
				else
				{
					const float4 v0 = *reinterpret_cast<const float4 *>(static_cast<const float *>(a.depth) + di);
					const float4 v1 = *reinterpret_cast<const float4 *>(static_cast<const float *>(a.depth) + di + 4);
					val[0] = v0.x; val[1] = v0.y; val[2] = v0.z; val[3] = v0.w;
					val[4] = v1.x; val[5] = v1.y; val[6] = v1.z; val[7] = v1.w;
				}
#pragma unroll
				for (int i = 0; i < 8; ++i)
					m[i] = (val[i] > a.min_depth && (a.max_depth == 0.0f || val[i] <= a.max_depth) && isfinite(val[i])) ? 255u : 0u;
			}
			uint2 mout;
			mout.x = m[0] | (m[1] << 8) | (m[2] << 16) | (m[3] << 24);
			mout.y = m[4] | (m[5] << 8) | (m[6] << 16) | (m[7] << 24);
			*reinterpret_cast<uint2 *>(mask + at) = mout;
			mall &= (m[0] & m[1]) | ((m[2] & m[3]) << 8) | ((m[4] & m[5]) << 16) | ((m[6] & m[7]) << 24);
		}
	}
	if (a.g.n_levels > 1)
	{
		const size_t at1 = a.g.off[1] + static_cast<size_t>(y1) * a.g.w[1] + 4 * xg;
		*reinterpret_cast<uint32_t *>(gray + at1) = static_cast<uint32_t>((sum[0] + 2) >> 2) | (static_cast<uint32_t>((sum[1] + 2) >> 2) << 8) |
		                                            (static_cast<uint32_t>((sum[2] + 2) >> 2) << 16) | (static_cast<uint32_t>((sum[3] + 2) >> 2) << 24);
		if (mask) *reinterpret_cast<uint32_t *>(mask + at1) = mall;
	}
}

// level l (>= 2) from level l-1
__global__ void orb_down_kernel(uint8_t * gray_all, uint8_t * mask_all, const OrbGeom g, int level)
{
	const int x = blockIdx.x * blockDim.x + threadIdx.x;
	const int y = blockIdx.y * blockDim.y + threadIdx.y;
	const int frame = blockIdx.z;
	if (x >= g.w[level] || y >= g.h[level]) return;
	uint8_t * gray = gray_all + static_cast<size_t>(frame) * g.frame_stride;
	const uint8_t * src = gray + g.off[level - 1];
	const int sw = g.w[level - 1];
	const int s = src[static_cast<size_t>(2 * y) * sw + 2 * x] + src[static_cast<size_t>(2 * y) * sw + 2 * x + 1] +
	              src[static_cast<size_t>(2 * y + 1) * sw + 2 * x] + src[static_cast<size_t>(2 * y + 1) * sw + 2 * x + 1];
	gray[g.off[level] + static_cast<size_t>(y) * g.w[level] + x] = static_cast<uint8_t>((s + 2) >> 2);
	if (mask_all)
	{
		uint8_t * mask = mask_all + static_cast<size_t>(frame) * g.frame_stride;
		const uint8_t * ms = mask + g.off[level - 1];
		const int m = ms[static_cast<size_t>(2 * y) * sw + 2 * x] & ms[static_cast<size_t>(2 * y) * sw + 2 * x + 1] &
		              ms[static_cast<size_t>(2 * y + 1) * sw + 2 * x] & ms[static_cast<size_t>(2 * y + 1) * sw + 2 * x + 1];
		mask[g.off[level] + static_cast<size_t>(y) * g.w[level] + x] = static_cast<uint8_t>(m);
	}
}

// ---- K2: FAST-9/16 score + 3x3 non-max suppression + border/mask filters -> candidate list --------
__device__ __forceinline__ int fast_score(const uint8_t * t, int stride, int thr)
{
	// t points at the pixel inside a shared tile; d[k] = centre - k-th pixel of the 16-pixel Bresenham circle
	// (OpenCV order: (0,3) (1,3) (2,2) (3,1) (3,0) (3,-1) (2,-2) (1,-3) (0,-3) (-1,-3) (-2,-2) (-3,-1) (-3,0) (-3,1) (-2,2) (-1,3))
	const int v = t[0];
	int d[16];
	d[0] = v - static_cast<int>(t[3 * stride]);
	d[1] = v - static_cast<int>(t[3 * stride + 1]);
	d[2] = v - static_cast<int>(t[2 * stride + 2]);
	d[3] = v - static_cast<int>(t[stride + 3]);
	d[4] = v - static_cast<int>(t[3]);
	d[5] = v - static_cast<int>(t[3 - stride]);
	d[6] = v - static_cast<int>(t[2 - 2 * stride]);
	d[7] = v - static_cast<int>(t[1 - 3 * stride]);
	d[8] = v - static_cast<int>(t[-3 * stride]);
	d[9] = v - static_cast<int>(t[-3 * stride - 1]);
	d[10] = v - static_cast<int>(t[-2 * stride - 2]);
	d[11] = v - static_cast<int>(t[-stride - 3]);
	d[12] = v - static_cast<int>(t[-3]);
	d[13] = v - static_cast<int>(t[stride - 3]);
	d[14] = v - static_cast<int>(t[2 * stride - 2]);
	d[15] = v - static_cast<int>(t[3 * stride - 1]);
	// every 9-arc contains pixel 0 or 8, and pixel 4 or 12: cheap rejection of flat neighbourhoods
	const bool reject = (abs(d[0]) <= thr && abs(d[8]) <= thr) || (abs(d[4]) <= thr && abs(d[12]) <= thr);
	int best = 0;
	if (!reject)
	{
		// cornerScore: max over the 16 arcs of 9 consecutive ring pixels of min(centre - pixel) (darker arcs) and of
		// min(pixel - centre) (brighter arcs).  Both polarities ride in one register as biased, strictly positive 16-bit
		// lanes, low = 256 + d, high = 256 - d (packed = d * (1 - 65536) + 0x01000100), and the minimum over each window of 9
		// comes from a doubling table (windows of 2, 4, 8, then one more element): 4 x 16 VIMNMX.U16x2 instead of 2 x 8 x 16.
		uint32_t p[16], q[16];
#pragma unroll
		for (int i = 0; i < 16; ++i) p[i] = static_cast<uint32_t>(d[i]) * 0xFFFF0001u + 0x01000100u;
#pragma unroll
		for (int i = 0; i < 16; ++i) q[i] = __vminu2(p[i], p[(i + 1) & 15]);          // windows of 2
		uint32_t r[16];
#pragma unroll
		for (int i = 0; i < 16; ++i) r[i] = __vminu2(q[i], q[(i + 2) & 15]);          // windows of 4
#pragma unroll
		for (int i = 0; i < 16; ++i) q[i] = __vminu2(r[i], r[(i + 4) & 15]);          // windows of 8
		uint32_t m = 0u;
#pragma unroll
		for (int i = 0; i < 16; ++i) m = __vmaxu2(m, __vminu2(q[i], p[(i + 8) & 15])); // windows of 9, maximum over the arcs
		best = static_cast<int>(max(m & 0xFFFFu, m >> 16)) - 256;
	}
	return best > thr ? best - 1 : 0;
}

// Fused FAST stage: score + 3x3 non-max suppression + border / mask filters -> candidate list, one 32x16 tile per CTA.
// The gray tile (4-pixel halo) is staged in shared memory; a cheap compass test (every 9-arc contains pixel 0 or 8 and
// pixel 4 or 12) compacts the few pixels that can be corners into a shared list, so the expensive arc minima run on
// dense warps instead of being dragged through every warp that holds one corner; the scores never leave shared memory.
constexpr int kFastTW = 32, kFastTH = 16;
__global__ void __launch_bounds__(256)
orb_fast_kernel(const uint8_t * __restrict__ gray_all, const uint8_t * __restrict__ mask_all, const OrbGeom g, int level,
                uint32_t * __restrict__ cand, int * __restrict__ cand_count)
{
	constexpr int GW = kFastTW + 8, GH = kFastTH + 8, SW = kFastTW + 2, SH = kFastTH + 2;
	__shared__ uint8_t s_gray[GH * GW];
	__shared__ uint8_t s_score[SH * SW];
	__shared__ uint16_t s_list[SH * SW];
	__shared__ int s_n;
	const int tid = threadIdx.x, lane = tid & 31;
	const int frame = blockIdx.z;
	const int w = g.w[level], h = g.h[level];
	const int x0 = blockIdx.x * kFastTW, y0 = blockIdx.y * kFastTH;
	const size_t plane = static_cast<size_t>(frame) * g.frame_stride + g.off[level];
	const uint8_t * img = gray_all + plane;
	for (int i = tid; i < GH * GW; i += 256)
	{
		const int gy = y0 - 4 + i / GW, gx = x0 - 4 + i % GW;
		s_gray[i] = (gx >= 0 && gx < w && gy >= 0 && gy < h) ? img[gy * w + gx] : 0;
	}
	for (int i = tid; i < SH * SW; i += 256) s_score[i] = 0;
	if (tid == 0) s_n = 0;
	__syncthreads();
	const int thr = g.fast_thr;
	// compass test over the tile + 1-pixel ring (the ring's scores feed the non-max suppression of the tile's edge)
	for (int i0 = 0; i0 < SH * SW; i0 += 256)
	{
		const int i = i0 + tid;
		bool maybe = false;
		if (i < SH * SW)
		{
			const int sy = i / SW - 1, sx = i % SW - 1;
			const int x = x0 + sx, y = y0 + sy;
			if (x >= 3 && x < w - 3 && y >= 3 && y < h - 3)
			{
				const uint8_t * t = s_gray + (sy + 4) * GW + sx + 4;
				const int v = t[0];
				const int d0 = abs(v - t[3 * GW]), d8 = abs(v - t[-3 * GW]), d4 = abs(v - t[3]), d12 = abs(v - t[-3]);
				maybe = !((d0 <= thr && d8 <= thr) || (d4 <= thr && d12 <= thr));
			}
		}
		const unsigned m = __ballot_sync(0xFFFFFFFFu, maybe);
		if (m)
		{
			int base = 0;
			if (lane == 0) base = atomicAdd(&s_n, __popc(m));
			base = __shfl_sync(0xFFFFFFFFu, base, 0);
			if (maybe) s_list[base + __popc(m & ((1u << lane) - 1u))] = static_cast<uint16_t>(i);
		}
	}
	__syncthreads();
	const int n_list = s_n;
	for (int k = tid; k < n_list; k += 256)
	{
		const int i = s_list[k];
		const int sy = i / SW - 1, sx = i % SW - 1;
		s_score[i] = static_cast<uint8_t>(fast_score(s_gray + (sy + 4) * GW + sx + 4, GW, thr));
	}
	__syncthreads();
	// 3x3 strict non-max suppression, KeyPointsFilter::runByPixelsMask and runByImageBorder
	const int slot = frame * g.n_levels + level;
	for (int i0 = 0; i0 < kFastTW * kFastTH; i0 += 256)
	{
		const int i = i0 + tid;
		const int ty = i / kFastTW, tx = i % kFastTW;
		const int x = x0 + tx, y = y0 + ty;
		bool keep = false;
		int sc0 = 0;
		if (x >= g.edge && x < w - g.edge && y >= g.edge && y < h - g.edge && x >= 3 && x < w - 3 && y >= 3 && y < h - 3)
		{
			const uint8_t * sc = s_score + (ty + 1) * SW + tx + 1;
			sc0 = sc[0];
			keep = sc0 > 0 && sc0 > sc[-SW - 1] && sc0 > sc[-SW] && sc0 > sc[-SW + 1] && sc0 > sc[-1] && sc0 > sc[1] && sc0 > sc[SW - 1] && sc0 > sc[SW] &&
			       sc0 > sc[SW + 1];
			if (keep && mask_all && mask_all[plane + static_cast<size_t>(y) * w + x] == 0) keep = false;
		}
		const unsigned m = __ballot_sync(0xFFFFFFFFu, keep);
		if (m)
		{
			int base = 0;
			if (lane == 0) base = atomicAdd(&cand_count[slot], __popc(m));
			base = __shfl_sync(0xFFFFFFFFu, base, 0);
			if (keep)
			{
				const int k = base + __popc(m & ((1u << lane) - 1u));
				if (k < kOrbCandCap) cand[static_cast<size_t>(slot) * kOrbCandCap + k] = (static_cast<uint32_t>(y * w + x) << 8) | static_cast<uint32_t>(sc0);
			}
		}
	}
}

// ---- K2 (TMA): the same stage with the gray tile + halo brought in by ONE cp.async.bulk.tensor (a 3-D tensor map over
// [frame][y][x] of the pyramid level; out-of-image pixels arrive as zeros, which is what the manual loop above stores), 64 x 32
// pixel tiles, and the per-pixel compass test and non-max suppression done four pixels at a time with byte-SIMD instructions
// (VABSDIFF4 / VSETGTU4): ~5 instead of ~25 instructions per pixel for the two full-tile passes.  Results are the same candidate
// SET (the selection kernel sorts it), bit for bit.
constexpr int kFastTmaTW = 64, kFastTmaTH = 32;
constexpr int kFastTmaGW = 96, kFastTmaGH = 40;   // staged box: x0-16 .. x0+80, y0-4 .. y0+36: the TMA needs a 16-byte aligned row start
                                                  // (x0 is a multiple of 64) and an inner extent that is a multiple of 16 bytes
constexpr int kFastTmaSW = 72, kFastTmaSH = 34;   // score plane: x0-4 .. x0+68, y0-1 .. y0+33

__device__ __forceinline__ void tma_load_3d(void * smem_dst, const void * tmap, int x, int y, int z, uint64_t * bar)
{
	asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(smem_u32(smem_dst)),
	             "l"(tmap), "r"(x), "r"(y), "r"(z), "r"(smem_u32(bar))
	             : "memory");
}

// Every lane reserves `cnt` consecutive slots of a shared-memory list: one atomic per warp.  All 32 lanes must call.
__device__ __forceinline__ int warp_reserve(int * counter, int cnt, int lane)
{
	int incl = cnt;
#pragma unroll
	for (int o = 1; o < 32; o <<= 1)
	{
		const int t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
		if (lane >= o) incl += t;
	}
	int base = 0;
	if (lane == 31 && incl) base = atomicAdd(counter, incl);
	base = __shfl_sync(0xFFFFFFFFu, base, 31);
	return base + incl - cnt;
}

struct alignas(64) OrbTensorMap
{
	unsigned long long opaque[16]; // CUtensorMap (128 bytes), filled by cuTensorMapEncodeTiled on the host
};

__global__ void __launch_bounds__(256)
orb_fast_tma_kernel(const __grid_constant__ OrbTensorMap tmap, const uint8_t * __restrict__ mask_all, const OrbGeom g, int level,
                    uint32_t * __restrict__ cand, int * __restrict__ cand_count)
{
	constexpr int GW = kFastTmaGW, GH = kFastTmaGH, SW = kFastTmaSW, SH = kFastTmaSH;
	__shared__ __align__(128) uint8_t s_gray[GH * GW];
	__shared__ __align__(16) uint8_t s_score[SH * SW];
	__shared__ __align__(16) uint16_t s_list[SH * (SW - 6)]; // compass survivors, then (as 32-bit words) the tile's output keys
	__shared__ int s_n;
	__shared__ __align__(8) uint64_t s_bar;
	const int tid = threadIdx.x, lane = tid & 31;
	const int frame = blockIdx.z;
	const int w = g.w[level], h = g.h[level];
	const int x0 = blockIdx.x * kFastTmaTW, y0 = blockIdx.y * kFastTmaTH;
	if (tid == 0)
	{
		mbar_init(&s_bar, 1);
		mbar_fence_init();
		s_n = 0;
	}
	for (int i = tid; i < SH * SW / 4; i += 256) reinterpret_cast<uint32_t *>(s_score)[i] = 0u;
	__syncthreads();
	if (tid == 0)
	{
		mbar_arrive_expect_tx(&s_bar, GW * GH);
		tma_load_3d(s_gray, &tmap, x0 - 16, y0 - 4, frame, &s_bar);
	}
	mbar_wait(&s_bar, 0);
	const int thr = g.fast_thr;
	const uint32_t thr4 = static_cast<uint32_t>(thr) * 0x01010101u;
	constexpr int WR = GW / 4;                                        // words per staged row
	const uint32_t * W = reinterpret_cast<const uint32_t *>(s_gray);
	// compass test (every 9-arc holds ring pixel 0 or 8, and 4 or 12), 4 pixels per item over the score plane
	for (int it0 = 0; it0 < SH * (SW / 4); it0 += 256) // whole warps iterate together: the list slots are reserved once per warp
	{
		const int it = it0 + tid;
		uint32_t maybe = 0u;
		int r = 0, k = 0;
		if (it < SH * (SW / 4))
		{
			r = it / (SW / 4), k = it % (SW / 4); // score row r = image row y0 - 1 + r; pixels x0 - 4 + 4k .. +3
			const int gy = r + 3;                 // staged row of the centre
			const int y = y0 - 1 + r, xb = x0 - 4 + 4 * k;
			// pixel x0 - 4 + 4k sits at staged column 4k + 12 = word k + 3
			const uint32_t wc = W[gy * WR + k + 3], wl = W[gy * WR + k + 2], wr = W[gy * WR + k + 4];
			const uint32_t up = W[(gy - 3) * WR + k + 3], dn = W[(gy + 3) * WR + k + 3];
			const uint32_t lf = __byte_perm(wl, wc, 0x4321), rt = __byte_perm(wc, wr, 0x6543);
			const uint32_t g0 = __vcmpgtu4(__vabsdiffu4(wc, dn), thr4), g8 = __vcmpgtu4(__vabsdiffu4(wc, up), thr4);
			const uint32_t g4 = __vcmpgtu4(__vabsdiffu4(wc, rt), thr4), g12 = __vcmpgtu4(__vabsdiffu4(wc, lf), thr4);
			maybe = (g0 | g8) & (g4 | g12);
			if (y < 3 || y >= h - 3) maybe = 0u;
			// only the tile and its 1-pixel ring are scored (x0 - 1 .. x0 + 64), inside the 3-pixel image margin of FAST
#pragma unroll
			for (int b = 0; b < 4; ++b)
			{
				const int x = xb + b;
				if (!(x >= 3 && x < w - 3 && x >= x0 - 1 && x <= x0 + kFastTmaTW)) maybe &= ~(0xFFu << (8 * b));
			}
		}
		const int cnt = __popc(maybe) >> 3; // the comparison masks are 0x00 / 0xFF per byte
		int at = warp_reserve(&s_n, cnt, lane);
#pragma unroll
		for (int b = 0; b < 4; ++b)
			if ((maybe >> (8 * b)) & 0xFFu) s_list[at++] = static_cast<uint16_t>(r * SW + 4 * k + b);
	}
	__syncthreads();
	const int n_list = s_n;
	for (int q = tid; q < n_list; q += 256)
	{
		const int i = s_list[q];
		const int r = i / SW, c = i % SW;
		s_score[i] = static_cast<uint8_t>(fast_score(s_gray + (r + 3) * GW + c + 12, GW, thr));
	}
	__syncthreads();
	// 3x3 strict non-max suppression + border / mask filters, 4 pixels per item over the tile
	const int slot = frame * g.n_levels + level;
	const size_t plane = static_cast<size_t>(frame) * g.frame_stride + g.off[level];
	const uint32_t * S = reinterpret_cast<const uint32_t *>(s_score); // 18 words per score row
	// survivors of the tile go to a shared list first (slots reserved once per warp), the mask test and the reservation in the frame's
	// global list then run over that list: one global atomic per 32 survivors instead of one per survivor, mask bytes loaded in parallel
	__syncthreads();
	if (tid == 0) s_n = 0;
	__syncthreads();
	uint32_t * s_out = reinterpret_cast<uint32_t *>(s_list); // <= 512 strict 3x3 maxima in a 64 x 32 tile; s_list holds 2244 u16
	for (int it0 = 0; it0 < kFastTmaTH * (kFastTmaTW / 4); it0 += 256)
	{
		const int it = it0 + tid;
		const int ty = it / (kFastTmaTW / 4), k = it % (kFastTmaTW / 4); // pixels x0 + 4k .. +3 of row y0 + ty
		const int y = y0 + ty, xb = x0 + 4 * k;
		const int sr = ty + 1;
		const uint32_t c = S[sr * 18 + k + 1];
		uint32_t keep = 0u;
		if (c != 0u && y >= g.edge && y < h - g.edge && y >= 3 && y < h - 3)
		{
			keep = __vcmpgtu4(c, 0u);
#pragma unroll
			for (int dr = -1; dr <= 1; ++dr)
			{
				const uint32_t a0 = S[(sr + dr) * 18 + k], a1 = S[(sr + dr) * 18 + k + 1], a2 = S[(sr + dr) * 18 + k + 2];
				keep &= __vcmpgtu4(c, __byte_perm(a0, a1, 0x6543)); // left neighbours
				keep &= __vcmpgtu4(c, __byte_perm(a1, a2, 0x4321)); // right neighbours
				if (dr != 0) keep &= __vcmpgtu4(c, a1);
			}
#pragma unroll
			for (int b = 0; b < 4; ++b)
			{
				const int x = xb + b;
				if (!(x >= g.edge && x < w - g.edge && x >= 3 && x < w - 3)) keep &= ~(0xFFu << (8 * b));
			}
		}
		const int cnt = __popc(keep) >> 3;
		int at = warp_reserve(&s_n, cnt, lane);
#pragma unroll
		for (int b = 0; b < 4; ++b)
			if ((keep >> (8 * b)) & 0xFFu) s_out[at++] = (static_cast<uint32_t>(y * w + xb + b) << 8) | ((c >> (8 * b)) & 0xFFu);
	}
	__syncthreads();
	const int n_out = s_n;
	for (int q0 = 0; q0 < n_out; q0 += 256)
	{
		const int q = q0 + tid;
		uint32_t key = 0u;
		bool ok = q < n_out;
		if (ok)
		{
			key = s_out[q];
			if (mask_all && mask_all[plane + (key >> 8)] == 0) ok = false;
		}
		const uint32_t m = __ballot_sync(0xFFFFFFFFu, ok);
		int base = 0;
		if (lane == 0 && m) base = atomicAdd(&cand_count[slot], __popc(m));
		base = __shfl_sync(0xFFFFFFFFu, base, 0);
		const int pos = base + __popc(m & ((1u << lane) - 1u));
		if (ok && pos < kOrbCandCap) cand[static_cast<size_t>(slot) * kOrbCandCap + pos] = key;
	}
}

// ---- K3: per (frame, level) selection: raster order, retainBest(2N) on FAST score, Harris, retainBest(N),
//          IC angle.  One CTA per frame, one launch per level; the two retainBest replays are block-cooperative
//          (partition_replay below). ----------------------------------------------------------------------
// Scratch of the block-cooperative replays below.
struct SelectScratch
{
	uint16_t * rpos; // [kOrbCandCap] positions of the right-hand scan's stops, by rank from the right
	int * warp_tot;  // [32]
	int * cut;       // [1]
};

// One Hoare-style partition pass over perm[lo..hi), replayed by the whole CTA.
//
// Both libstdc++ loops this file replays (std::__unguarded_partition and the bidirectional std::__partition)
// have the same shape: a left cursor that walks up and STOPS at elements with stop_l(x), a right cursor that walks
// down and stops at elements with stop_r(x), the two stopped elements are swapped and both cursors move on; the
// loop ends when the cursors meet.  Because each cursor only ever visits positions the other has not touched
// yet, the k-th stop of either cursor is the k-th element (from its side) of the ORIGINAL array that satisfies its
// predicate, and pair k is swapped iff L_k < R_k (monotone in k).  So the sequential result is: swap (L_k, R_k) for
// all k with L_k < R_k, and the left cursor ends at min(first unswapped L, last swapped R).  Ranks come from one
// block-wide prefix sum; every thread owns a contiguous segment of <= 32 positions (kOrbCandCap / kOrbSelectThreads).
// Returns the final left cursor (INT_MAX if neither exists).  All threads must call; result is uniform.
template <class StopL, class StopR>
__device__ inline int partition_replay(uint16_t * perm, const float * resp, int lo, int hi, const SelectScratch & sc, StopL stop_l, StopR stop_r)
{
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
	const int len = hi - lo;
	const int seg = (len + static_cast<int>(blockDim.x) - 1) / static_cast<int>(blockDim.x);
	const int b = lo + tid * seg, e = min(b + seg, hi);
	uint32_t ml = 0, mr = 0;
	for (int i = b; i < e; ++i)
	{
		const float x = resp[perm[i]];
		ml |= (stop_l(x) ? 1u : 0u) << (i - b);
		mr |= (stop_r(x) ? 1u : 0u) << (i - b);
	}
	// block exclusive scan of (count_l | count_r << 16)
	const int mine = __popc(ml) | (__popc(mr) << 16);
	int incl = mine;
#pragma unroll
	for (int o = 1; o < 32; o <<= 1)
	{
		const int t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
		if (lane >= o) incl += t;
	}
	if (lane == 31) sc.warp_tot[warp] = incl;
	if (tid == 0) *sc.cut = 0x7FFFFFFF;
	__syncthreads();
	int pre = 0, total = 0;
	for (int w = 0; w < nwarps; ++w)
	{
		const int t = sc.warp_tot[w];
		if (w < warp) pre += t;
		total += t;
	}
	const int ex = pre + incl - mine;
	const int ex_l = ex & 0xFFFF, ex_r = ex >> 16, tot_r = total >> 16;
	{
		int r = tot_r - 1 - ex_r; // rank from the right of this segment's first right-stop
		for (uint32_t m = mr; m; m &= m - 1)
		{
			sc.rpos[r] = static_cast<uint16_t>(b + __ffs(m) - 1);
			--r;
		}
	}
	__syncthreads();
	{
		int k = ex_l;
		int best = 0x7FFFFFFF;
		for (uint32_t m = ml; m; m &= m - 1, ++k)
		{
			const int i = b + __ffs(m) - 1;
			const int j = k < tot_r ? static_cast<int>(sc.rpos[k]) : -1;
			if (i < j)
			{
				const uint16_t t = perm[i];
				perm[i] = perm[j];
				perm[j] = t;
				best = min(best, j);
			}
			else best = min(best, i);
		}
		if (best != 0x7FFFFFFF) atomicMin(sc.cut, best);
	}
	__syncthreads();
	const int cut = *sc.cut;
	__syncthreads(); // *sc.cut is re-armed by the next call
	return cut;
}

// libstdc++ std::nth_element(first, nth, last, greater-by-response) on perm[first..last): introselect with the
// median-of-three pivot moved to `first`, __unguarded_partition on [first+1, last), insertion sort of the last <= 3.
// Called by all threads of the CTA; thread 0 does the O(1) steps.
__device__ inline void nth_element_replay(uint16_t * perm, const float * resp, int first, int nth, int last, const SelectScratch & sc)
{
	if (first == last || nth == last) return;
	auto comp = [&](int a, int b) { return resp[perm[a]] > resp[perm[b]]; };
	auto swp = [&](int a, int b) {
		const uint16_t t = perm[a];
		perm[a] = perm[b];
		perm[b] = t;
	};
	int depth = 2 * (31 - __clz(last - first));
	while (last - first > 3)
	{
		if (depth == 0)
		{
			// __heap_select fallback of introselect: cannot occur before 2*log2(n) unbalanced partitions;
			// a plain selection keeps the SET right even then (order parity is lost, flagged by the tests)
			if (threadIdx.x == 0)
				for (int i = first; i <= nth; ++i)
				{
					int b = i;
					for (int j = i + 1; j < last; ++j)
						if (comp(j, b)) b = j;
					swp(i, b);
				}
			__syncthreads();
			return;
		}
		--depth;
		if (threadIdx.x == 0)
		{
			// __move_median_to_first(first, first+1, mid, last-1)
			const int r = first, a = first + 1, b = first + (last - first) / 2, c = last - 1;
			if (comp(a, b))
			{
				if (comp(b, c)) swp(r, b);
				else if (comp(a, c)) swp(r, c);
				else swp(r, a);
			}
			else if (comp(a, c)) swp(r, a);
			else if (comp(b, c)) swp(r, c);
			else swp(r, b);
		}
		__syncthreads();
		const float pv = resp[perm[first]];
		// __unguarded_partition(first+1, last, pivot): left stops at !(x > pv), right at !(pv > x)
		const int cut = partition_replay(perm, resp, first + 1, last, sc, [pv](float x) { return !(x > pv); }, [pv](float x) { return !(pv > x); });
		if (cut <= nth) first = cut;
		else last = cut;
	}
	if (threadIdx.x == 0)
	{
		// __insertion_sort(first, last)
		for (int i = first + 1; i < last; ++i)
		{
			const uint16_t val = perm[i];
			const float rv = resp[val];
			if (rv > resp[perm[first]])
			{
				for (int j = i; j > first; --j) perm[j] = perm[j - 1];
				perm[first] = val;
			}
			else
			{
				int j = i;
				while (rv > resp[perm[j - 1]])
				{
					perm[j] = perm[j - 1];
					--j;
				}
				perm[j] = val;
			}
		}
	}
	__syncthreads();
}

// KeyPointsFilter::retainBest(keypoints, n_points): returns the new size.  Called by all threads of the CTA.
__device__ inline int retain_best_replay(uint16_t * perm, const float * resp, int n, int n_points, const SelectScratch & sc)
{
	if (n_points < 0 || n <= n_points) return n;
	if (n_points == 0) return 0;
	nth_element_replay(perm, resp, 0, n_points - 1, n, sc);
	const float amb = resp[perm[n_points - 1]];
	// std::partition(perm + n_points, perm + n, response >= amb) (bidirectional version): left stops at
	// !(x >= amb), right stops at x >= amb; the result is n_points + #{x >= amb}
	int keep = 0;
	{
		// count first (the partition below permutes positions, not values, so the count is order-free)
		__shared__ int s_keep;
		if (threadIdx.x == 0) s_keep = 0;
		__syncthreads();
		int c = 0;
		for (int i = n_points + threadIdx.x; i < n; i += blockDim.x) c += resp[perm[i]] >= amb ? 1 : 0;
		if (c) atomicAdd(&s_keep, c);
		__syncthreads();
		keep = s_keep;
		__syncthreads();
	}
	partition_replay(perm, resp, n_points, n, sc, [amb](float x) { return !(x >= amb); }, [amb](float x) { return x >= amb; });
	return n_points + keep;
}

__device__ __forceinline__ float fast_atan2_deg(float y, float x)
{
	const float K = static_cast<float>(180.0 / 3.141592653589793238462643383279502884197169399375);
	const float p1 = __fmul_rn(0.9997878412794807f, K), p3 = __fmul_rn(-0.3258083974640975f, K), p5 = __fmul_rn(0.1555786518463281f, K),
	            p7 = __fmul_rn(-0.04432655554792128f, K);
	const float ax = fabsf(x), ay = fabsf(y);
	const float eps = static_cast<float>(2.220446049250313e-16);
	float a, c, c2;
	if (ax >= ay)
	{
		c = __fdiv_rn(ay, __fadd_rn(ax, eps));
		c2 = __fmul_rn(c, c);
		a = __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(p7, c2), p5), c2), p3), c2), p1), c);
	}
	else
	{
		c = __fdiv_rn(ax, __fadd_rn(ay, eps));
		c2 = __fmul_rn(c, c);
		a = __fsub_rn(90.f, __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(p7, c2), p5), c2), p3), c2), p1), c));
	}
	if (x < 0) a = __fsub_rn(180.f, a);
	if (y < 0) a = __fsub_rn(360.f, a);
	return a;
}

struct OrbSelectArgs
{
	const uint8_t * gray;
	OrbGeom g;
	const uint32_t * cand;
	const int * cand_count;
	OrbKeypoint * level_kp; // [n_frames][n_levels][level_cap]
	int * level_n;          // [n_frames][n_levels]
	int level_cap;
	int * overflow;         // set when a candidate list had to be truncated
	int level;              // pyramid level this launch handles (one launch per level: shared memory is sized per level)
	int cand_cap;           // candidates of this level kept in shared memory (<= kOrbCandCap)
};

__global__ void __launch_bounds__(kOrbSelectThreads)
orb_select_kernel(const OrbSelectArgs a)
{
	extern __shared__ __align__(16) unsigned char smem_raw[];
	const int ccap = a.cand_cap;
	uint32_t * keys = reinterpret_cast<uint32_t *>(smem_raw);   // [ccap]
	float * resp = reinterpret_cast<float *>(keys + ccap);        // [ccap]
	uint16_t * perm = reinterpret_cast<uint16_t *>(resp + ccap);  // [ccap]
	__shared__ int s_warp_tot[32], s_cut;
	const SelectScratch sc{perm + ccap, s_warp_tot, &s_cut};
	__shared__ int s_umax[20];

	const int tid = threadIdx.x;
	const int level = a.level, frame = blockIdx.x;
	const int slot = frame * a.g.n_levels + level;
	const int w = a.g.w[level], h = a.g.h[level];
	const uint8_t * img = a.gray + static_cast<size_t>(frame) * a.g.frame_stride + a.g.off[level];
	int n = a.cand_count[slot];
	if (n > ccap)
	{
		n = ccap;
		if (tid == 0) atomicExch(a.overflow, 1);
	}
	for (int i = tid; i < n; i += blockDim.x) keys[i] = a.cand[static_cast<size_t>(slot) * kOrbCandCap + i];
	if (tid == 0)
	{
		// umax table of the circular patch (ORB computeKeyPoints)
		const int half = a.g.patch / 2;
		const int vmax = static_cast<int>(floorf(half * sqrtf(2.f) / 2 + 1));
		const int vmin = static_cast<int>(ceilf(half * sqrtf(2.f) / 2));
		for (int v = 0; v <= vmax; ++v) s_umax[v] = static_cast<int>(rint(sqrt(static_cast<double>(half) * half - static_cast<double>(v) * v)));
		for (int v = half, v0 = 0; v >= vmin; --v)
		{
			while (s_umax[v0] == s_umax[v0 + 1]) ++v0;
			s_umax[v] = v0;
			++v0;
		}
	}
	__syncthreads();
	// raster order (FAST emits keypoints row by row).  Every candidate is a different pixel, so its place in raster order is the number
	// of candidates at smaller positions: a position bitmap (in the not yet used response array) + one block-wide prefix sum of its
	// popcounts replaces a 105-stage bitonic sort of 16k keys.
	{
		// (a static array for the segment prefixes would push the CTA past the 196 KB shared-memory carve-out and halve the L1 left for
		// the Harris / angle patches: everything lives in the dynamic allocation)
		const int nw_max = ccap - ccap / 8;
		uint32_t * bits = reinterpret_cast<uint32_t *>(resp);   // 7/8 of the response array: 32 * nw_max positions per pass
		int * s_seg = reinterpret_cast<int *>(bits + nw_max);   // exclusive popcount prefix of every 8-word segment of the bitmap
		uint32_t * sorted = reinterpret_cast<uint32_t *>(perm); // perm + rpos: ccap words
		const int lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
		constexpr int kSegPerThread = kOrbCandCap / 8 / kOrbSelectThreads; // 8-word segments owned by a thread
		const int n_pos = w * h;
		int base = 0;
		for (int p0 = 0; p0 < n_pos; p0 += 32 * nw_max)
		{
			const int nw = min(nw_max, (n_pos - p0 + 31) >> 5);
			for (int i = tid; i < nw; i += blockDim.x) bits[i] = 0u;
			__syncthreads();
			for (int i = tid; i < n; i += blockDim.x)
			{
				const int rel = static_cast<int>(keys[i] >> 8) - p0;
				if (rel >= 0 && rel < 32 * nw) atomicOr(&bits[rel >> 5], 1u << (rel & 31));
			}
			__syncthreads();
			int tot[kSegPerThread], tsum = 0;
#pragma unroll
			for (int k = 0; k < kSegPerThread; ++k)
			{
				const int w0 = (tid * kSegPerThread + k) * 8;
				int c = 0;
				for (int j = w0; j < min(w0 + 8, nw); ++j) c += __popc(bits[j]);
				tot[k] = c;
				tsum += c;
			}
			int incl = tsum;
#pragma unroll
			for (int o = 1; o < 32; o <<= 1)
			{
				const int t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
				if (lane >= o) incl += t;
			}
			if (lane == 31) s_warp_tot[warp] = incl;
			__syncthreads();
			int pre = 0, total = 0;
			for (int q = 0; q < nwarps; ++q)
			{
				const int t = s_warp_tot[q];
				if (q < warp) pre += t;
				total += t;
			}
			int ex = pre + incl - tsum;
#pragma unroll
			for (int k = 0; k < kSegPerThread; ++k)
			{
				if ((tid * kSegPerThread + k) * 8 < nw) s_seg[tid * kSegPerThread + k] = ex;
				ex += tot[k];
			}
			__syncthreads();
			for (int i = tid; i < n; i += blockDim.x)
			{
				const uint32_t key = keys[i];
				const int rel = static_cast<int>(key >> 8) - p0;
				if (rel >= 0 && rel < 32 * nw)
				{
					const int wi = rel >> 5;
					int r = base + s_seg[wi >> 3] + __popc(bits[wi] & ((1u << (rel & 31)) - 1u));
					for (int j = wi & ~7; j < wi; ++j) r += __popc(bits[j]);
					sorted[r] = key;
				}
			}
			base += total;
			__syncthreads();
		}
		for (int i = tid; i < n; i += blockDim.x) keys[i] = sorted[i];
		__syncthreads();
	}
	for (int i = tid; i < n; i += blockDim.x)
	{
		resp[i] = static_cast<float>(keys[i] & 0xFFu);
		perm[i] = static_cast<uint16_t>(i);
	}
	__syncthreads();
	const int n_level = a.g.n_per_level[level];
	int m = retain_best_replay(perm, resp, n, 2 * n_level, sc);
	// Harris responses of the kept candidates (HarrisResponses, blockSize 7, k 0.04)
	for (int i = tid; i < m; i += blockDim.x)
	{
		const int pos = static_cast<int>(keys[perm[i]] >> 8);
		const int x0 = pos % w, y0 = pos / w;
		int A = 0, B = 0, Cc = 0;
		if (x0 >= 4 && x0 < w - 4 && y0 >= 4 && y0 < h - 4)
		{
			// the 9x9 neighbourhood once into registers (81 loads instead of 8 per position of the 7x7 block)
			int pt[9][9];
#pragma unroll
			for (int r = 0; r < 9; ++r)
#pragma unroll
				for (int c = 0; c < 9; ++c) pt[r][c] = img[(y0 - 4 + r) * w + x0 - 4 + c];
#pragma unroll
			for (int r = 1; r <= 7; ++r)
#pragma unroll
				for (int c = 1; c <= 7; ++c)
				{
					const int Ix = (pt[r][c + 1] - pt[r][c - 1]) * 2 + (pt[r - 1][c + 1] - pt[r - 1][c - 1]) + (pt[r + 1][c + 1] - pt[r + 1][c - 1]);
					const int Iy = (pt[r + 1][c] - pt[r - 1][c]) * 2 + (pt[r + 1][c - 1] - pt[r - 1][c - 1]) + (pt[r + 1][c + 1] - pt[r - 1][c + 1]);
					A += Ix * Ix;
					B += Iy * Iy;
					Cc += Ix * Iy;
				}
		}
		else
		for (int dy = -3; dy <= 3; ++dy)
			for (int dx = -3; dx <= 3; ++dx)
			{
				const int x = x0 + dx, y = y0 + dy;
				const int xm = reflect101(x - 1, w), xp = reflect101(x + 1, w), ym = reflect101(y - 1, h), yp = reflect101(y + 1, h);
				const int xc = reflect101(x, w), yc = reflect101(y, h);
				const int p00 = img[ym * w + xm], p01 = img[ym * w + xc], p02 = img[ym * w + xp];
				const int p10 = img[yc * w + xm], p12 = img[yc * w + xp];
				const int p20 = img[yp * w + xm], p21 = img[yp * w + xc], p22 = img[yp * w + xp];
				const int Ix = (p12 - p10) * 2 + (p02 - p00) + (p22 - p20);
				const int Iy = (p21 - p01) * 2 + (p20 - p00) + (p22 - p02);
				A += Ix * Ix;
				B += Iy * Iy;
				Cc += Ix * Iy;
			}
		const float scale = __fdiv_rn(1.f, __fmul_rn(static_cast<float>(4 * 7), 255.f));
		const float s4 = __fmul_rn(__fmul_rn(__fmul_rn(scale, scale), scale), scale);
		const float fa = static_cast<float>(A), fb = static_cast<float>(B), fc = static_cast<float>(Cc);
		const float t3 = __fadd_rn(fa, fb);
		resp[perm[i]] = __fmul_rn(__fsub_rn(__fsub_rn(__fmul_rn(fa, fb), __fmul_rn(fc, fc)), __fmul_rn(__fmul_rn(0.04f, t3), t3)), s4);
	}
	__syncthreads();
	const int kept = retain_best_replay(perm, resp, m, n_level, sc);
	m = min(kept, a.level_cap);
	if (tid == 0)
	{
		a.level_n[slot] = m;
		if (kept > a.level_cap) atomicExch(a.overflow, 1);
	}
	// IC angle + output: one warp per keypoint, lane = column of the circular patch, so that a row of the patch is one coalesced load and
	// the 31 rows are independent loads in flight (a thread per keypoint walked ~700 dependent byte loads).  The moments are integer sums:
	// any summation order gives the reference's value.
	const int half = a.g.patch / 2;
	const float sf = static_cast<float>(1 << level);
	const int lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
	// rows of the circular patch that hold column u = lane - half: |v| <= vlim (umax is non-increasing in v); -1 = column outside the patch
	const int u_lane = lane - half;
	int vlim = -1;
	if (u_lane <= half)
		for (int v = 0; v <= half; ++v)
			if ((v == 0 ? half : s_umax[v]) >= (u_lane < 0 ? -u_lane : u_lane)) vlim = v;
	for (int i = warp; i < m; i += nwarps)
	{
		const uint32_t key = keys[perm[i]];
		const int pos = static_cast<int>(key >> 8);
		const int x0 = pos % w, y0 = pos / w;
		int m01 = 0, m10 = 0;
		if (half <= 15 && x0 >= half && x0 < w - half && y0 >= half && y0 < h - half)
		{
			// default patch, keypoint away from the border (always, with the default edge threshold): lane = column u, rows |v| <= vlim(u)
			const uint8_t * col = img + y0 * w + x0 + u_lane;
			int sum = 0;
#pragma unroll
			for (int v = -15; v <= 15; ++v)
				if ((v < 0 ? -v : v) <= vlim)
				{
					const int val = col[v * w];
					sum += val;
					m01 += v * val;
				}
			m10 = u_lane * sum;
		}
		else
		for (int ub = -half; ub <= half; ub += 32) // one trip for the default 31-pixel patch
		{
			const int u = ub + lane;
			const int xx = reflect101(x0 + u, w);
#pragma unroll 4
			for (int v = -half; v <= half; ++v)
			{
				const int d = v == 0 ? half : s_umax[v < 0 ? -v : v];
				if (u <= half && u >= -d && u <= d)
				{
					const int val = img[reflect101(y0 + v, h) * w + xx];
					m10 += u * val;
					m01 += v * val;
				}
			}
		}
		m10 = __reduce_add_sync(0xFFFFFFFFu, m10);
		m01 = __reduce_add_sync(0xFFFFFFFFu, m01);
		if (lane == 0)
		{
			OrbKeypoint kp;
			kp.x = __fmul_rn(static_cast<float>(x0), sf);
			kp.y = __fmul_rn(static_cast<float>(y0), sf);
			kp.size = __fmul_rn(static_cast<float>(a.g.patch), sf);
			kp.angle = fast_atan2_deg(static_cast<float>(m01), static_cast<float>(m10));
			kp.response = resp[perm[i]];
			kp.octave = level;
			a.level_kp[static_cast<size_t>(slot) * a.level_cap + i] = kp;
		}
	}
}

// ---- K4: concatenate the levels of a frame and apply Feature2D::limitKeypoints -----------------------
__global__ void __launch_bounds__(1024)
orb_merge_kernel(const OrbKeypoint * __restrict__ level_kp, const int * __restrict__ level_n, int n_levels, int level_cap, int max_features,
                 OrbKeypoint * __restrict__ out, int * __restrict__ out_n, int out_cap)
{
	extern __shared__ __align__(16) unsigned char smem_raw[];
	unsigned long long * skey = reinterpret_cast<unsigned long long *>(smem_raw); // [pad]
	__shared__ int s_off[kOrbMaxLevels + 1];
	const int frame = blockIdx.x, tid = threadIdx.x;
	if (tid == 0)
	{
		s_off[0] = 0;
		for (int l = 0; l < n_levels; ++l) s_off[l + 1] = s_off[l] + level_n[frame * n_levels + l];
	}
	__syncthreads();
	const int total = s_off[n_levels];
	auto src = [&](int i) -> const OrbKeypoint & {
		int l = 0;
		while (i >= s_off[l + 1]) ++l;
		return level_kp[(static_cast<size_t>(frame) * n_levels + l) * level_cap + (i - s_off[l])];
	};
	if (max_features <= 0 || total <= max_features)
	{
		const int n = min(total, out_cap);
		for (int i = tid; i < n; i += blockDim.x) out[static_cast<size_t>(frame) * out_cap + i] = src(i);
		if (tid == 0) out_n[frame] = n;
		return;
	}
	// multimap<fabs(response), index> walked in reverse: strongest first, later index first among equals
	int pad = 1;
	while (pad < total) pad <<= 1;
	for (int i = tid; i < pad; i += blockDim.x)
	{
		unsigned long long k = 0ull; // sorts last in descending order
		if (i < total)
		{
			const float r = fabsf(src(i).response);
			k = (static_cast<unsigned long long>(__float_as_uint(r)) << 32) | static_cast<unsigned>(i + 1);
		}
		skey[i] = k;
	}
	__syncthreads();
	for (int k = 2; k <= pad; k <<= 1)
		for (int j = k >> 1; j > 0; j >>= 1)
		{
			for (int idx = tid; idx < pad; idx += blockDim.x)
			{
				const int ixj = idx ^ j;
				if (ixj > idx)
				{
					const unsigned long long x = skey[idx], y = skey[ixj];
					if ((x < y) == ((idx & k) == 0)) // descending
					{
						skey[idx] = y;
						skey[ixj] = x;
					}
				}
			}
			__syncthreads();
		}
	const int n = min(max_features, out_cap);
	for (int i = tid; i < n; i += blockDim.x) out[static_cast<size_t>(frame) * out_cap + i] = src(static_cast<int>(skey[i] & 0xFFFFFFFFull) - 1);
	if (tid == 0) out_n[frame] = n;
}

// ---- K5: 7x7 sigma=2 blur of every level (float sepFilter2D semantics) -------------------------------
__constant__ float kOrbGauss7[7];

constexpr int kBlurTW = 32, kBlurTH = 16;

__global__ void __launch_bounds__(256)
orb_blur_kernel(const uint8_t * __restrict__ gray_all, uint8_t * __restrict__ blur_all, const OrbGeom g, int level)
{
	// gray tile with a 3-pixel reflect-101 halo -> shared memory, row pass into floats, column pass; every pixel of the
	// level is read from global memory ~1.6 times instead of once per tap
	__shared__ uint8_t s_g[kBlurTH + 6][kBlurTW + 8];
	__shared__ float rowf[kBlurTH + 6][kBlurTW];
	const int frame = blockIdx.z;
	const int w = g.w[level], h = g.h[level];
	const uint8_t * img = gray_all + static_cast<size_t>(frame) * g.frame_stride + g.off[level];
	uint8_t * out = blur_all + static_cast<size_t>(frame) * g.frame_stride + g.off[level];
	const int x0 = blockIdx.x * kBlurTW, y0 = blockIdx.y * kBlurTH;
	const int tid = threadIdx.x;
	for (int i = tid; i < (kBlurTH + 6) * (kBlurTW + 6); i += 256)
	{
		const int ry = i / (kBlurTW + 6), rx = i % (kBlurTW + 6);
		const int y = reflect101(min(y0 + ry - 3, h + 2), h), x = reflect101(min(x0 + rx - 3, w + 2), w);
		s_g[ry][rx] = img[y * w + x];
	}
	__syncthreads();
	// row pass (plain order, fused multiply-add) for the TH+6 rows the column pass needs
	for (int i = tid; i < (kBlurTH + 6) * kBlurTW; i += 256)
	{
		const int ry = i / kBlurTW, rx = i % kBlurTW;
		float s = __fmul_rn(static_cast<float>(s_g[ry][rx]), kOrbGauss7[0]);
#pragma unroll
		for (int k = 1; k < 7; ++k) s = __fmaf_rn(static_cast<float>(s_g[ry][rx + k]), kOrbGauss7[k], s);
		rowf[ry][rx] = s;
	}
	__syncthreads();
	// column pass (symmetric, fused multiply-add), then saturate_cast<uchar> (round half to even)
	const int tx = tid % kBlurTW;
	for (int ty = tid / kBlurTW; ty < kBlurTH; ty += 256 / kBlurTW)
	{
		const int x = x0 + tx, y = y0 + ty;
		if (x >= w || y >= h) continue;
		const int c = ty + 3;
		float s = __fmul_rn(rowf[c][tx], kOrbGauss7[3]);
#pragma unroll
		for (int k = 1; k <= 3; ++k) s = __fmaf_rn(__fadd_rn(rowf[c + k][tx], rowf[c - k][tx]), kOrbGauss7[3 + k], s);
		int v = __float2int_rn(s);
		v = v < 0 ? 0 : (v > 255 ? 255 : v);
		out[static_cast<size_t>(y) * w + x] = static_cast<uint8_t>(v);
	}
}

// ---- K5 (TMA): the same blur on the 64 x 32 tiles / 96 x 40 staged boxes of the FAST kernel (one cp.async.bulk.tensor per CTA, same
// tensor map).  The TMA fills out-of-image pixels with zeros; border tiles rewrite their 3-pixel halo with the reflect-101 values.  Both
// passes keep a sliding window in registers: a thread produces 8 consecutive outputs of a row (14 bytes in, from 4 aligned words), then 8
// consecutive outputs of a column (14 floats in) -- ~30 instead of ~200 instructions per pixel, same float operations in the same order.
__global__ void __launch_bounds__(256)
orb_blur_tma_kernel(const __grid_constant__ OrbTensorMap tmap, uint8_t * __restrict__ blur_all, const OrbGeom g, int level)
{
	constexpr int GW = kFastTmaGW, GH = kFastTmaGH, TW = kFastTmaTW, TH = kFastTmaTH;
	constexpr int RH = TH + 6; // rows of the row pass: y0 - 3 .. y0 + TH + 2
	__shared__ __align__(128) uint8_t s_gray[GH * GW];
	__shared__ __align__(16) float s_row[RH * TW];
	__shared__ __align__(8) uint64_t s_bar;
	const int tid = threadIdx.x;
	const int frame = blockIdx.z;
	const int w = g.w[level], h = g.h[level];
	const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;
	if (tid == 0)
	{
		mbar_init(&s_bar, 1);
		mbar_fence_init();
	}
	__syncthreads();
	if (tid == 0)
	{
		mbar_arrive_expect_tx(&s_bar, GW * GH);
		tma_load_3d(s_gray, &tmap, x0 - 16, y0 - 4, frame, &s_bar);
	}
	mbar_wait(&s_bar, 0);
	if (x0 < 3 || x0 + TW + 3 > w || y0 < 3 || y0 + TH + 3 > h)
	{
		// image pixel (x, y) sits at staged (x - x0 + 16, y - y0 + 4); columns first (rows of the image), then whole rows
		for (int i = tid; i < GH * (TW + 6); i += 256)
		{
			const int ry = i / (TW + 6), x = x0 - 3 + i % (TW + 6), y = y0 - 4 + ry;
			if (y >= 0 && y < h && (x < 0 || (x >= w && x <= w + 2))) s_gray[ry * GW + x - x0 + 16] = s_gray[ry * GW + reflect101(x, w) - x0 + 16];
		}
		__syncthreads();
		for (int i = tid; i < RH * (TW + 6); i += 256)
		{
			const int ry = 1 + i / (TW + 6), cx = 13 + i % (TW + 6), y = y0 - 4 + ry;
			if (y < 0 || (y >= h && y <= h + 2)) s_gray[ry * GW + cx] = s_gray[(reflect101(y, h) - y0 + 4) * GW + cx];
		}
		__syncthreads();
	}
	const float k0 = kOrbGauss7[0], k1 = kOrbGauss7[1], k2 = kOrbGauss7[2], k3 = kOrbGauss7[3], k4 = kOrbGauss7[4], k5 = kOrbGauss7[5],
	            k6 = kOrbGauss7[6];
	// row pass (plain order, fused multiply-add): outputs x0 + 8j .. + 7 of staged row r + 1 read staged columns 8j + 13 .. 8j + 26
	for (int it = tid; it < RH * (TW / 8); it += 256)
	{
		const int r = it >> 3, j = it & 7;
		const uint32_t * wp = reinterpret_cast<const uint32_t *>(s_gray + (r + 1) * GW) + 2 * j + 3;
		const uint32_t w0 = wp[0], w1 = wp[1], w2 = wp[2], w3 = wp[3];
		float p[14];
		p[0] = static_cast<float>((w0 >> 8) & 0xFFu);
		p[1] = static_cast<float>((w0 >> 16) & 0xFFu);
		p[2] = static_cast<float>(w0 >> 24);
		p[3] = static_cast<float>(w1 & 0xFFu);
		p[4] = static_cast<float>((w1 >> 8) & 0xFFu);
		p[5] = static_cast<float>((w1 >> 16) & 0xFFu);
		p[6] = static_cast<float>(w1 >> 24);
		p[7] = static_cast<float>(w2 & 0xFFu);
		p[8] = static_cast<float>((w2 >> 8) & 0xFFu);
		p[9] = static_cast<float>((w2 >> 16) & 0xFFu);
		p[10] = static_cast<float>(w2 >> 24);
		p[11] = static_cast<float>(w3 & 0xFFu);
		p[12] = static_cast<float>((w3 >> 8) & 0xFFu);
		p[13] = static_cast<float>((w3 >> 16) & 0xFFu);
		float o[8];
#pragma unroll
		for (int q = 0; q < 8; ++q)
		{
			float s = __fmul_rn(p[q], k0);
			s = __fmaf_rn(p[q + 1], k1, s);
			s = __fmaf_rn(p[q + 2], k2, s);
			s = __fmaf_rn(p[q + 3], k3, s);
			s = __fmaf_rn(p[q + 4], k4, s);
			s = __fmaf_rn(p[q + 5], k5, s);
			s = __fmaf_rn(p[q + 6], k6, s);
			o[q] = s;
		}
		float4 * dst = reinterpret_cast<float4 *>(s_row + r * TW + 8 * j);
		dst[0] = make_float4(o[0], o[1], o[2], o[3]);
		dst[1] = make_float4(o[4], o[5], o[6], o[7]);
	}
	__syncthreads();
	// column pass (symmetric, fused multiply-add), saturate_cast<uchar> (round half to even): column c, output rows 8 rg .. 8 rg + 7
	const int c = tid & (TW - 1), rg = tid >> 6;
	const int x = x0 + c;
	if (x >= w) return;
	float v[14];
#pragma unroll
	for (int k = 0; k < 14; ++k) v[k] = s_row[(8 * rg + k) * TW + c];
	uint8_t * out = blur_all + static_cast<size_t>(frame) * g.frame_stride + g.off[level];
#pragma unroll
	for (int q = 0; q < 8; ++q)
	{
		const int y = y0 + 8 * rg + q;
		float s = __fmul_rn(v[q + 3], k3);
		s = __fmaf_rn(__fadd_rn(v[q + 4], v[q + 2]), k4, s);
		s = __fmaf_rn(__fadd_rn(v[q + 5], v[q + 1]), k5, s);
		s = __fmaf_rn(__fadd_rn(v[q + 6], v[q]), k6, s);
		int iv = __float2int_rn(s);
		iv = iv < 0 ? 0 : (iv > 255 ? 255 : iv);
		if (y < h) out[static_cast<size_t>(y) * w + x] = static_cast<uint8_t>(iv);
	}
}

// ---- K6: steered BRIEF (computeOrbDescriptors, WTA_K = 2) --------------------------------------------
constexpr int kOrbDescribeKp = 32;  // keypoints per CTA of the describe kernel

__global__ void __launch_bounds__(256)
orb_describe_kernel(const uint8_t * __restrict__ gray_all, const uint8_t * __restrict__ blur_all, const OrbGeom g,
                    const OrbKeypoint * __restrict__ kps, const int * __restrict__ n_kp, int cap, uint8_t * __restrict__ desc)
{
	// phase 1: the rotation of each keypoint once per keypoint (double-precision cos / sin rounded to float, as
	// computeOrbDescriptors does), phase 2: one thread per (keypoint, descriptor byte)
	// the 256 test locations as floats in shared memory: lanes of a warp read DIFFERENT tests (byte = lane), which the
	// constant cache would serialise 32 ways
	__shared__ float4 s_pat[256];
	__shared__ float s_ca[kOrbDescribeKp], s_sa[kOrbDescribeKp];
	__shared__ int s_cx[kOrbDescribeKp], s_cy[kOrbDescribeKp], s_level[kOrbDescribeKp];
	const int frame = blockIdx.y;
	const int kp0 = blockIdx.x * kOrbDescribeKp;
	const int n = min(n_kp[frame] - kp0, kOrbDescribeKp);
	if (n <= 0) return;
	for (int i = threadIdx.x; i < 256; i += blockDim.x)
		s_pat[i] = make_float4(static_cast<float>(kOrbPattern31[4 * i]), static_cast<float>(kOrbPattern31[4 * i + 1]),
		                       static_cast<float>(kOrbPattern31[4 * i + 2]), static_cast<float>(kOrbPattern31[4 * i + 3]));
	for (int i = threadIdx.x; i < n; i += blockDim.x)
	{
		const OrbKeypoint kp = kps[static_cast<size_t>(frame) * cap + kp0 + i];
		const float scale = __fdiv_rn(1.f, static_cast<float>(1 << kp.octave));
		const float angle = __fmul_rn(kp.angle, static_cast<float>(3.141592653589793238462643383279502884197169399375 / 180.0));
		s_ca[i] = static_cast<float>(cos(static_cast<double>(angle)));
		s_sa[i] = static_cast<float>(sin(static_cast<double>(angle)));
		s_cx[i] = __float2int_rn(__fmul_rn(kp.x, scale));
		s_cy[i] = __float2int_rn(__fmul_rn(kp.y, scale));
		s_level[i] = kp.octave;
	}
	__syncthreads();
	for (int t = threadIdx.x; t < n * 32; t += blockDim.x)
	{
		const int ki = t >> 5, byte = t & 31;
		const int level = s_level[ki];
		const int w = g.w[level], h = g.h[level];
		const uint8_t * raw = gray_all + static_cast<size_t>(frame) * g.frame_stride + g.off[level];
		const uint8_t * blr = blur_all + static_cast<size_t>(frame) * g.frame_stride + g.off[level];
		const float ca = s_ca[ki], sa = s_sa[ki];
		const int cx = s_cx[ki], cy = s_cy[ki];
		// rotated taps reach at most ceil(13 * sqrt(2)) = 19 pixels from the centre: keypoints further than that from every
		// border (almost all of them) skip the bounds test
		const bool inside = cx >= 19 && cy >= 19 && cx < w - 19 && cy < h - 19;
		auto tap = [&](float px, float py) -> int {
			const float fx = __fsub_rn(__fmul_rn(px, ca), __fmul_rn(py, sa));
			const float fy = __fadd_rn(__fmul_rn(px, sa), __fmul_rn(py, ca));
			const int x = cx + __float2int_rn(fx), y = cy + __float2int_rn(fy);
			if (inside || (x >= 0 && x < w && y >= 0 && y < h)) return blr[y * w + x];
			return raw[reflect101(y, h) * w + reflect101(x, w)]; // unblurred reflected border
		};
		int val = 0;
#pragma unroll
		for (int b = 0; b < 8; ++b)
		{
			const float4 p = s_pat[byte * 8 + b];
			const int t0 = tap(p.x, p.y), t1 = tap(p.z, p.w);
			val |= (t0 < t1) << b;
		}
		desc[(static_cast<size_t>(frame) * cap + kp0 + ki) * 32 + byte] = static_cast<uint8_t>(val);
	}
}

// ---- K6 (patch): the same descriptors with the 39 x 39 blurred patch of every keypoint staged in shared memory first (aligned
// 32-bit loads, ~100 sectors per keypoint instead of 512 scattered byte gathers), one warp per keypoint.  Needs every rotated tap inside
// the level (edge threshold >= 19, the default 31 is) and rows that are a multiple of 4 bytes; the caller falls back to the kernel above.
constexpr int kOrbPatchR = 19, kOrbPatchPitch = 48;

__global__ void __launch_bounds__(256)
orb_describe_patch_kernel(const uint8_t * __restrict__ blur_all, const OrbGeom g, const OrbKeypoint * __restrict__ kps, const int * __restrict__ n_kp,
                          int cap, uint8_t * __restrict__ desc)
{
	__shared__ float4 s_pat[256];
	__shared__ __align__(16) uint8_t s_patch[8][(2 * kOrbPatchR + 1) * kOrbPatchPitch];
	__shared__ float s_ca[kOrbDescribeKp], s_sa[kOrbDescribeKp];
	__shared__ int s_cx[kOrbDescribeKp], s_cy[kOrbDescribeKp], s_level[kOrbDescribeKp];
	const int frame = blockIdx.y;
	const int kp0 = blockIdx.x * kOrbDescribeKp;
	const int n = min(n_kp[frame] - kp0, kOrbDescribeKp);
	if (n <= 0) return;
	// test t = 8 * byte + bit is kept at [bit * 32 + byte]: the 32 lanes of a warp (lane = descriptor byte) read consecutive float4
	for (int i = threadIdx.x; i < 256; i += blockDim.x)
		s_pat[(i & 7) * 32 + (i >> 3)] = make_float4(static_cast<float>(kOrbPattern31[4 * i]), static_cast<float>(kOrbPattern31[4 * i + 1]),
		                                             static_cast<float>(kOrbPattern31[4 * i + 2]), static_cast<float>(kOrbPattern31[4 * i + 3]));
	// the rotation of each keypoint once per keypoint, 32 keypoints per warp instruction (double-precision cos / sin: computed by every
	// lane of the keypoint's warp it would be the whole cost of the kernel)
	for (int i = threadIdx.x; i < n; i += blockDim.x)
	{
		const OrbKeypoint kp = kps[static_cast<size_t>(frame) * cap + kp0 + i];
		const float scale = __fdiv_rn(1.f, static_cast<float>(1 << kp.octave));
		const float angle = __fmul_rn(kp.angle, static_cast<float>(3.141592653589793238462643383279502884197169399375 / 180.0));
		s_ca[i] = static_cast<float>(cos(static_cast<double>(angle)));
		s_sa[i] = static_cast<float>(sin(static_cast<double>(angle)));
		s_cx[i] = __float2int_rn(__fmul_rn(kp.x, scale));
		s_cy[i] = __float2int_rn(__fmul_rn(kp.y, scale));
		s_level[i] = kp.octave;
	}
	__syncthreads();
	const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	uint8_t * patch = s_patch[warp];
	for (int ki = warp; ki < n; ki += 8)
	{
		const float ca = s_ca[ki], sa = s_sa[ki];
		const int cx = s_cx[ki], cy = s_cy[ki];
		const int level = s_level[ki];
		const int w = g.w[level];
		const uint8_t * blr = blur_all + static_cast<size_t>(frame) * g.frame_stride + g.off[level];
		const int xa = (cx - kOrbPatchR) & ~3;                 // aligned column of the first staged word
		const int n_words = ((cx + kOrbPatchR) >> 2) - (xa >> 2) + 1; // <= 11
		__syncwarp();
		for (int idx = lane; idx < (2 * kOrbPatchR + 1) * 11; idx += 32)
		{
			const int r = idx / 11, j = idx - r * 11;
			if (j < n_words)
				reinterpret_cast<uint32_t *>(patch + r * kOrbPatchPitch)[j] =
					*reinterpret_cast<const uint32_t *>(blr + static_cast<size_t>(cy - kOrbPatchR + r) * w + xa + 4 * j);
		}
		__syncwarp();
		const uint8_t * centre = patch + kOrbPatchR * kOrbPatchPitch + (cx - xa);
		int val = 0;
#pragma unroll
		for (int b = 0; b < 8; ++b)
		{
			const float4 p = s_pat[b * 32 + lane];
			const int x0 = __float2int_rn(__fsub_rn(__fmul_rn(p.x, ca), __fmul_rn(p.y, sa)));
			const int y0 = __float2int_rn(__fadd_rn(__fmul_rn(p.x, sa), __fmul_rn(p.y, ca)));
			const int x1 = __float2int_rn(__fsub_rn(__fmul_rn(p.z, ca), __fmul_rn(p.w, sa)));
			const int y1 = __float2int_rn(__fadd_rn(__fmul_rn(p.z, sa), __fmul_rn(p.w, ca)));
			const int t0 = centre[y0 * kOrbPatchPitch + x0], t1 = centre[y1 * kOrbPatchPitch + x1];
			val |= (t0 < t1) << b;
		}
		desc[(static_cast<size_t>(frame) * cap + kp0 + ki) * 32 + lane] = static_cast<uint8_t>(val);
	}
}

// ---- K7: generateKeypoints3DDepth (depth the size of the image, one camera, identity local transform) ---
struct OrbXyzArgs
{
	const void * depth;
	int depth_type, w, h;
	float fx, fy, cx, cy, min_depth, max_depth;
	const OrbKeypoint * kps;
	const int * n_kp;
	int cap;
	float * xyz;
};

__device__ __forceinline__ float depth_at(const void * depth, int type, size_t base, int w, int v, int u)
{
	if (type == 1)
	{
		const unsigned short d = static_cast<const unsigned short *>(depth)[base + static_cast<size_t>(v) * w + u];
		return (d > 0 && d < 65535) ? __fmul_rn(static_cast<float>(d), 0.001f) : 0.0f;
	}
	return static_cast<const float *>(depth)[base + static_cast<size_t>(v) * w + u];
}

__global__ void orb_xyz_kernel(const OrbXyzArgs a)
{
	const int frame = blockIdx.y;
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= a.n_kp[frame]) return;
	const OrbKeypoint kp = a.kps[static_cast<size_t>(frame) * a.cap + i];
	float * out = a.xyz + (static_cast<size_t>(frame) * a.cap + i) * 3;
	const float nan = __int_as_float(0x7FC00000);
	out[0] = out[1] = out[2] = nan;
	if (!a.depth) return;
	const size_t base = static_cast<size_t>(frame) * a.w * a.h;
	const float x = kp.x, y = kp.y;
	int u = static_cast<int>(__fadd_rn(x, 0.5f)), v = static_cast<int>(__fadd_rn(y, 0.5f));
	if (u == a.w && x < static_cast<float>(a.w)) u = a.w - 1;
	if (v == a.h && y < static_cast<float>(a.h)) v = a.h - 1;
	if (!(u >= 0 && u < a.w && v >= 0 && v < a.h)) return;
	float depth = depth_at(a.depth, a.depth_type, base, a.w, v, u);
	if (depth == 0.0f || !isfinite(depth)) return;
	// util2d::getDepth smoothing: 3x3 window, neighbours within 2 % of the centre, weights 4/2/1
	float sumWeights = 0.f, sumDepths = 0.f;
	const float depthError = __fmul_rn(0.02f, depth);
	for (int uu = max(u - 1, 0); uu <= min(u + 1, a.w - 1); ++uu)
		for (int vv = max(v - 1, 0); vv <= min(v + 1, a.h - 1); ++vv)
		{
			if (uu == u && vv == v) continue;
			float d = depth_at(a.depth, a.depth_type, base, a.w, vv, uu);
			if (d != 0.0f && isfinite(d) && fabsf(__fsub_rn(d, depth)) < depthError)
			{
				if (uu == u || vv == v)
				{
					sumWeights = __fadd_rn(sumWeights, 2.0f);
					d = __fmul_rn(d, 2.0f);
				}
				else sumWeights = __fadd_rn(sumWeights, 1.0f);
				sumDepths = __fadd_rn(sumDepths, d);
			}
		}
	depth = __fmul_rn(depth, 4.0f);
	sumWeights = __fadd_rn(sumWeights, 4.0f);
	depth = __fdiv_rn(__fadd_rn(depth, sumDepths), sumWeights);
	if (!(depth > 0.0f)) return;
	const float cx = a.cx > 0.0f ? a.cx : __fsub_rn(static_cast<float>(a.w / 2), 0.5f);
	const float cy = a.cy > 0.0f ? a.cy : __fsub_rn(static_cast<float>(a.h / 2), 0.5f);
	const float px = __fdiv_rn(__fmul_rn(__fsub_rn(x, cx), depth), a.fx);
	const float py = __fdiv_rn(__fmul_rn(__fsub_rn(y, cy), depth), a.fy);
	if ((a.min_depth < 0.0f || depth > a.min_depth) && (a.max_depth <= 0.0f || depth <= a.max_depth))
	{
		out[0] = px;
		out[1] = py;
		out[2] = depth;
	}
}

// keypoint coordinates as a plain float2 array (the TO side of the verification kernels)
__global__ void orb_uv_kernel(const OrbKeypoint * __restrict__ kps, const int * __restrict__ n_kp, int cap, float * __restrict__ uv)
{
	const int frame = blockIdx.y;
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= cap) return;
	const size_t o = static_cast<size_t>(frame) * cap + i;
	const bool ok = i < n_kp[frame];
	uv[2 * o] = ok ? kps[o].x : 0.f;
	uv[2 * o + 1] = ok ? kps[o].y : 0.f;
}

} // namespace lcd
