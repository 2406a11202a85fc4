// =====================================================================================================
// raster.h — the small rasteriser of the end-to-end tests.  TEST INFRASTRUCTURE ONLY, shared by oracle/_ref/librefshader.so
// (driver.cpp: after the reference's own mesh and vertex shaders) and tests/mesh_stage_host.cpp (after their restatement).
// =====================================================================================================
#pragma once

#include "../../include/niagara_cull.h"

#include <math.h>
#include <stdint.h>
#include <stddef.h>

#include <algorithm>
#include <utility>

// ---- a small reference rasteriser for end-to-end tests (OURS, not the reference's: Vulkan's fixed function) --------------
// Facing as the mesh shader's own MESH_CULL code decides it (meshlet.mesh.glsl:154,175-181): in the y-up screen space
// (clip.xy / clip.w * 0.5 + 0.5) * screen a triangle is front facing iff eb.x * ec.y > eb.y * ec.x (= the pipeline's
// COUNTER_CLOCKWISE front face + BACK culling, shaders.cpp:687-688).  Pixels are placed with the reference's flipped
// viewport {0, height, width, -height} (niagara.cpp:1641): row = (0.5 - 0.5 * ndc.y) * height, which is also the uv
// convention of projectSphere's aabb (math.h:19).  A triangle with a corner at w <= 0 is skipped (no near clipping);
// samples at pixel centres, inclusive edges; depth = clip.z / clip.w interpolated affinely, test GREATER (reverse Z, clear 0).
// mode 0: depth[] = max(depth[], triangle depth).   mode 1: depth[] is read-only; slot_hit[slot] = 1 when some covered sample of
// the slot has exactly the stored depth (i.e. the slot owns or ties a pixel of the final image).

// one triangle given as three clip-space corners; returns true when (mode 1) a covered sample has exactly the stored depth
inline bool rasterTriangle(const float* const corner[3], uint32_t width, uint32_t height, float* depth, int mode)
{
	double sx[3], sy[3], sz[3];
	for (int c = 0; c < 3; ++c)
	{
		const float* p = corner[c];
		if (!(p[3] > 0.0f))
			return false;
		float fx = (p[0] / p[3] * 0.5f + 0.5f) * float(width), fy = (p[1] / p[3] * 0.5f + 0.5f) * float(height);
		sx[c] = fx;
		sy[c] = fy;
		sz[c] = double(p[2] / p[3]);
	}
	double ebx = sx[1] - sx[0], eby = sy[1] - sy[0], ecx = sx[2] - sx[0], ecy = sy[2] - sy[0];
	double area = ebx * ecy - eby * ecx;
	if (!(area > 0.0))
		return false; // back facing or zero area
	// flipped viewport: rows count from the top; swapping two corners keeps the edge functions positive inside
	for (int c = 0; c < 3; ++c)
		sy[c] = double(height) - sy[c];
	std::swap(sx[1], sx[2]);
	std::swap(sy[1], sy[2]);
	std::swap(sz[1], sz[2]);
	double minx = std::min(sx[0], std::min(sx[1], sx[2])), maxx = std::max(sx[0], std::max(sx[1], sx[2]));
	double miny = std::min(sy[0], std::min(sy[1], sy[2])), maxy = std::max(sy[0], std::max(sy[1], sy[2]));
	if (!(maxx >= 0.0 && maxy >= 0.0 && minx <= double(width) && miny <= double(height)))
		return false;
	int x0 = int(std::max(0.0, floor(minx - 0.5))), x1 = int(std::min(double(width) - 1.0, ceil(maxx - 0.5)));
	int y0 = int(std::max(0.0, floor(miny - 0.5))), y1 = int(std::min(double(height) - 1.0, ceil(maxy - 0.5)));
	bool hit = false;
	for (int y = y0; y <= y1; ++y)
		for (int x = x0; x <= x1; ++x)
		{
			double px = x + 0.5, py = y + 0.5;
			double w0 = (sx[1] - px) * (sy[2] - py) - (sy[1] - py) * (sx[2] - px);
			double w1 = (sx[2] - px) * (sy[0] - py) - (sy[2] - py) * (sx[0] - px);
			double w2 = (sx[0] - px) * (sy[1] - py) - (sy[0] - py) * (sx[1] - px);
			if (w0 < 0.0 || w1 < 0.0 || w2 < 0.0)
				continue;
			float z = float((w0 * sz[0] + w1 * sz[1] + w2 * sz[2]) / (w0 + w1 + w2));
			float& d = depth[size_t(y) * width + x];
			if (mode == 0)
			{
				if (z > d)
					d = z;
			}
			else if (z == d)
				hit = true;
		}
	return hit;
}

// every triangle of `slots` mesh-stage outputs (records[slot] = {vertexCount, triangleCount, ...}, positions[slot][64][4],
// triangles[slot][96][3]); mode as rasterTriangle, slot_hit[slot] = 1 when one of the slot's triangles owns / ties a pixel
inline int rasterizeSlots(const float* positions, const uint8_t* triangles, const uint32_t* records, uint32_t slots, uint32_t width, uint32_t height, float* depth,
    uint8_t* slot_hit, int mode)
{
	for (uint32_t slot = 0; slot < slots; ++slot)
	{
		uint32_t vc = records[slot * 4 + 0], tc = records[slot * 4 + 1];
		for (uint32_t t = 0; t < tc && t < 96; ++t)
		{
			const float* corner[3];
			for (int c = 0; c < 3; ++c)
			{
				uint32_t v = triangles[(size_t(slot) * 96 + t) * 3 + c];
				if (v >= vc)
					return NVC_ERROR_INVALID_ARGUMENT;
				corner[c] = positions + (size_t(slot) * 64 + v) * 4;
			}
			if (rasterTriangle(corner, width, height, depth, mode) && slot_hit)
				slot_hit[slot] = 1;
		}
	}
	return NVC_OK;
}
