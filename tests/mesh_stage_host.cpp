// TEST INFRASTRUCTURE: the vertex work of the reference's meshlet.mesh.glsl and mesh.vert.glsl restated for the host, with the
// arithmetic of the product's raster_depth_kernel (strict IEEE, GLSL operation order: rotateQuat, * scale + position,
// projection * (view * vec4(wpos, 1))), followed by the test rasteriser (oracle/refshader/raster.h).  It has the C interface of
// those entry points of oracle/_ref/librefshader.so: tests/refshader_lib.py loads it where the reference's shaders cannot be
// built and holds its outputs to the reference's pinned ones.  Built by refshader_lib.py with g++ -ffp-contract=off into
// tests/_build/ (git-ignored).
#include "../oracle/refshader/raster.h"

#include <string.h>

namespace
{

struct V3
{
	float x, y, z;
};

// GLSL float16_t -> float: exact, subnormals included
float half_to_float(uint16_t h)
{
	uint32_t s = uint32_t(h & 0x8000u) << 16, e = (h >> 10) & 31u, m = h & 0x3ffu, bits;
	if (e == 31)
		bits = s | 0x7f800000u | (m << 13);
	else if (e)
		bits = s | ((e + 112) << 23) | (m << 13);
	else
	{
		float f = float(m) * 0x1p-24f;
		memcpy(&bits, &f, 4);
		bits |= s;
	}
	float f;
	memcpy(&f, &bits, 4);
	return f;
}

V3 cross3(V3 a, V3 b)
{
	return { a.y * b.z - b.y * a.z, a.z * b.x - b.z * a.x, a.x * b.y - b.x * a.y };
}

// math.h rotateQuat: v + 2 * cross(q.xyz, cross(q.xyz, v) + q.w * v)
V3 rotate_quat(V3 v, const float q[4])
{
	V3 qv = { q[0], q[1], q[2] };
	V3 c1 = cross3(qv, v);
	V3 t = { c1.x + q[3] * v.x, c1.y + q[3] * v.y, c1.z + q[3] * v.z };
	V3 c2 = cross3(qv, t);
	return { v.x + 2.0f * c2.x, v.y + 2.0f * c2.y, v.z + 2.0f * c2.z };
}

// GLSL mat4 * vec4, column-major: ((col0 * x + col1 * y) + col2 * z) + col3 * w
void mat4_mul_vec4(const float* m, const float v[4], float out[4])
{
	for (int r = 0; r < 4; ++r)
		out[r] = m[r] * v[0] + m[4 + r] * v[1] + m[8 + r] * v[2] + m[12 + r] * v[3];
}

// gl_Position of vertex vi of draw d
void clip_position(const float* projection, const float* view, const NvcMeshDraw& d, const NvcVertex& vx, float clip[4])
{
	V3 r = rotate_quat({ half_to_float(vx.vx), half_to_float(vx.vy), half_to_float(vx.vz) }, d.orientation);
	float w[4] = { r.x * d.scale + d.position[0], r.y * d.scale + d.position[1], r.z * d.scale + d.position[2], 1.0f };
	float v[4];
	mat4_mul_vec4(view, w, v);
	mat4_mul_vec4(projection, v, clip);
}

struct Inputs
{
	const float* projection;
	const NvcCullData* pass;
	const NvcMeshTaskCommand* commands;
	size_t command_count;
	const NvcMeshDraw* draws;
	size_t draw_count;
	const NvcMeshlet* meshlets;
	size_t meshlet_count;
	const uint8_t* meshletdata;
	size_t meshletdata_bytes;
	const NvcVertex* vertices;
	size_t vertex_count;
};

// one mesh workgroup (meshlet.mesh.glsl main) for cluster index ci: records {vertexCount, triangleCount, drawId or ~0, 0},
// positions[64][4], triangles[96][3]; false when the cluster refers outside the inputs
bool mesh_group(const Inputs& in, uint32_t ci, uint32_t* record, float* positions, uint8_t* triangles)
{
	record[0] = record[1] = record[3] = 0;
	record[2] = ~0u;
	if (ci == ~0u)
		return true; // SetMeshOutputsEXT(0, 0)
	if ((ci & 0xffffffu) >= in.command_count)
		return false;
	const NvcMeshTaskCommand& command = in.commands[ci & 0xffffffu];
	const uint32_t mi = command.taskOffset + (ci >> 24);
	if (mi >= in.meshlet_count || command.drawId >= in.draw_count)
		return false;
	const NvcMeshlet& ml = in.meshlets[mi];
	const NvcMeshDraw& draw = in.draws[command.drawId];
	const uint32_t vc = ml.vertexCount, tc = ml.triangleCount;
	const size_t index_offset = size_t(ml.dataOffset) + (ml.shortRefs == 1 ? (vc + 1) / 2 : vc);
	if (vc > 64 || tc > 96 || (index_offset * 4 + size_t(tc) * 3) > in.meshletdata_bytes)
		return false;
	record[0] = vc;
	record[1] = tc;
	record[2] = vc ? command.drawId : ~0u;
	for (uint32_t i = 0; i < vc; ++i)
	{
		uint32_t ref;
		if (ml.shortRefs == 1)
		{
			uint16_t r16;
			memcpy(&r16, in.meshletdata + size_t(ml.dataOffset) * 4 + size_t(i) * 2, 2);
			ref = r16;
		}
		else
			memcpy(&ref, in.meshletdata + (size_t(ml.dataOffset) + i) * 4, 4);
		const uint32_t vi = ref + ml.baseVertex;
		if (vi >= in.vertex_count)
			return false;
		clip_position(in.projection, in.pass->view, draw, in.vertices[vi], positions + i * 4);
	}
	memcpy(triangles, in.meshletdata + index_offset * 4, size_t(tc) * 3);
	return true;
}

Inputs inputs(const float* projection16, const NvcCullData* pass, const void* task_commands, size_t commands_bytes, const void* draws, size_t draws_bytes,
    const void* meshlets, size_t meshlets_bytes, const void* meshletdata, size_t meshletdata_bytes, const void* vertices, size_t vertices_bytes)
{
	return { projection16, pass, static_cast<const NvcMeshTaskCommand*>(task_commands), commands_bytes / sizeof(NvcMeshTaskCommand), static_cast<const NvcMeshDraw*>(draws),
		draws_bytes / sizeof(NvcMeshDraw), static_cast<const NvcMeshlet*>(meshlets), meshlets_bytes / sizeof(NvcMeshlet), static_cast<const uint8_t*>(meshletdata), meshletdata_bytes,
		static_cast<const NvcVertex*>(vertices), vertices_bytes / sizeof(NvcVertex) };
}

} // namespace

extern "C"
{

// the mesh stage over the (X, Y, Z) grid of ccb: slot x + 256 * y + 16 * z reads cib[slot]
int rs_mesh_clusters(const float* projection16, const NvcCullData* pass, float, float, const void* task_commands, size_t commands_bytes, const void* draws,
    size_t draws_bytes, const void* meshlets, size_t meshlets_bytes, const void* meshletdata, size_t meshletdata_bytes, const void* vertices, size_t vertices_bytes,
    const uint32_t* cluster_indices, size_t cib_bytes, const uint32_t* cluster_count4, uint32_t* records, float* positions, uint8_t* triangles, int)
{
	const Inputs in = inputs(projection16, pass, task_commands, commands_bytes, draws, draws_bytes, meshlets, meshlets_bytes, meshletdata, meshletdata_bytes, vertices, vertices_bytes);
	for (uint32_t z = 0; z < cluster_count4[3]; ++z)
		for (uint32_t y = 0; y < cluster_count4[2]; ++y)
			for (uint32_t x = 0; x < cluster_count4[1]; ++x)
			{
				const size_t slot = size_t(x) + size_t(y) * 256 + size_t(z) * 16;
				if ((slot + 1) * 4 > cib_bytes || !mesh_group(in, cluster_indices[slot], records + slot * 4, positions + slot * 256, triangles + slot * 288))
					return NVC_ERROR_INVALID_ARGUMENT;
			}
	return NVC_OK;
}

// task-shading mode: the i-th mesh workgroup of command c reads payloads[c].clusterIndices[i] into slot first_slot[c] + i
int rs_mesh_payloads(const float* projection16, const NvcCullData* pass, float, float, const void* task_commands, size_t commands_bytes, uint32_t command_count,
    const void* draws, size_t draws_bytes, const void* meshlets, size_t meshlets_bytes, const void* meshletdata, size_t meshletdata_bytes, const void* vertices,
    size_t vertices_bytes, const NvcMeshTaskPayload* payloads, const uint32_t* emit_counts, const uint32_t* first_slot, uint32_t* records, float* positions,
    uint8_t* triangles, int)
{
	const Inputs in = inputs(projection16, pass, task_commands, commands_bytes, draws, draws_bytes, meshlets, meshlets_bytes, meshletdata, meshletdata_bytes, vertices, vertices_bytes);
	for (uint32_t c = 0; c < command_count; ++c)
		for (uint32_t i = 0; i < emit_counts[c] && i < NVC_TASK_WGSIZE; ++i)
		{
			const size_t slot = size_t(first_slot[c]) + i;
			if (!mesh_group(in, payloads[c].clusterIndices[i], records + slot * 4, positions + slot * 256, triangles + slot * 288))
				return NVC_ERROR_INVALID_ARGUMENT;
			records[slot * 4 + 3] = c;
		}
	return NVC_OK;
}

int rs_rasterize(const float* positions, const uint8_t* triangles, const uint32_t* records, uint32_t slots, uint32_t width, uint32_t height, float* depth,
    uint8_t* slot_hit, int mode)
{
	return rasterizeSlots(positions, triangles, records, slots, width, height, depth, slot_hit, mode);
}

// the draw path: mesh.vert.glsl for every index of every command (gl_DrawIDARB = i), triangles rasterised as they come
int rs_draw_indexed(const float* projection16, const NvcCullData* pass, float, float, const void* draw_commands, size_t commands_bytes, uint32_t command_count,
    const void* draws, size_t draws_bytes, const void* vertices, size_t vertices_bytes, const uint32_t* indices, size_t index_count, uint32_t width, uint32_t height,
    float* depth, uint8_t* command_hit, int mode)
{
	const NvcMeshDrawCommand* cmds = static_cast<const NvcMeshDrawCommand*>(draw_commands);
	const NvcMeshDraw* mesh_draws = static_cast<const NvcMeshDraw*>(draws);
	const NvcVertex* verts = static_cast<const NvcVertex*>(vertices);
	if (size_t(command_count) * sizeof(NvcMeshDrawCommand) > commands_bytes)
		return NVC_ERROR_INVALID_ARGUMENT;
	for (uint32_t i = 0; i < command_count; ++i)
	{
		const NvcMeshDrawCommand& c = cmds[i];
		if (uint64_t(c.firstIndex) + c.indexCount > index_count || (c.drawId + 1) * sizeof(NvcMeshDraw) > draws_bytes)
			return NVC_ERROR_INVALID_ARGUMENT;
		for (uint32_t inst = 0; inst < c.instanceCount; ++inst)
			for (uint32_t t = 0; t + 2 < c.indexCount; t += 3)
			{
				float clip[3][4];
				const float* corner[3];
				for (int k = 0; k < 3; ++k)
				{
					const uint32_t vi = indices[c.firstIndex + t + k] + c.vertexOffset;
					if ((size_t(vi) + 1) * sizeof(NvcVertex) > vertices_bytes)
						return NVC_ERROR_INVALID_ARGUMENT;
					clip_position(projection16, pass->view, mesh_draws[c.drawId], verts[vi], clip[k]);
					corner[k] = clip[k];
				}
				if (rasterTriangle(corner, width, height, depth, mode) && command_hit)
					command_hit[i] = 1;
			}
	}
	return NVC_OK;
}

} // extern "C"
