// =====================================================================================================
// driver.cpp — runs the reference's own shaders (compiled through glsl_shim.h, see gen.py) on host arrays.
// TEST INFRASTRUCTURE ONLY (oracle/_ref/librefshader.so).  It plays the part of niagara.cpp's frame loop for
// the visibility path: the buffer fills, descriptor bindings, push constants and dispatch sizes below restate
//   cull lambda      niagara.cpp:1530-1574   fill(dccb,0,4) -> drawcull (ceil(drawCount/64) groups) -> tasksubmit (1 group)
//   render lambda    niagara.cpp:1582-1610   fill(ccb,0,4)  -> clustercull (indirect dccb+4)       -> clustersubmit (1 group)
//   task submission  niagara.cpp:1666-1679   vkCmdDrawMeshTasksIndirectEXT(dccb+4) with meshlet.task
//   pyramid lambda   niagara.cpp:1703-1733   per mip: depthreduce over ceil(w/32) x ceil(h/32) groups
// Workgroups of one dispatch are spread over host threads (the shaders' atomics are real atomics); the invocations
// of a workgroup run in ascending gl_LocalInvocationIndex order on one thread, as fibers when the shader uses
// barrier().  Output order therefore differs from run to run exactly as on a GPU; compare as sets.
// =====================================================================================================
#include "../../include/niagara_cull.h"
#include "glsl_shim.h"
#include "raster.h"
#include "rs_shader.h"

#include <stdio.h>
#include <ucontext.h>

#include <algorithm>
#include <atomic>
#include <functional>
#include <thread>
#include <vector>

namespace glsl
{
thread_local uvec3 gl_GlobalInvocationID, gl_LocalInvocationID, gl_WorkGroupID;
thread_local uint gl_LocalInvocationIndex;
thread_local MeshPerVertex gl_MeshVerticesEXT[256];
thread_local uvec3 gl_PrimitiveTriangleIndicesEXT[256];
thread_local MeshPerPrimitive gl_MeshPrimitivesEXT[256];
thread_local int gl_VertexIndex, gl_DrawIDARB;
thread_local vec4 gl_Position;
} // namespace glsl

extern const RsShader rs_shader_drawcull, rs_shader_tasksubmit, rs_shader_clustercull, rs_shader_clustersubmit, rs_shader_depthreduce, rs_shader_meshlet_task, rs_shader_meshlet_mesh, rs_shader_mesh_vert;

namespace
{

using glsl::uint;

// ---- fibers: one per invocation of a workgroup whose shader calls barrier() ---------------------------------------
struct Fiber
{
	ucontext_t ctx;
	std::vector<char> stack;
	bool done = false;
};

thread_local ucontext_t* t_scheduler = nullptr;
thread_local Fiber* t_current = nullptr;
thread_local void (*t_main)() = nullptr;
thread_local uint t_emit[3];
thread_local uint t_mesh_outputs[2];

void fiberEntry()
{
	t_main();
	t_current->done = true;
	swapcontext(&t_current->ctx, t_scheduler);
}

void setInvocation(const uint* ls, uint gx, uint gy, uint gz, uint lx, uint ly, uint lz)
{
	glsl::gl_WorkGroupID = glsl::uvec3(gx, gy, gz);
	glsl::gl_LocalInvocationID = glsl::uvec3(lx, ly, lz);
	glsl::gl_GlobalInvocationID = glsl::uvec3(gx * ls[0] + lx, gy * ls[1] + ly, gz * ls[2] + lz);
	glsl::gl_LocalInvocationIndex = (lz * ls[1] + ly) * ls[0] + lx;
}

void runGroup(const RsShader& s, uint gx, uint gy, uint gz)
{
	const uint* ls = s.local_size;
	uint count = ls[0] * ls[1] * ls[2];
	if (!s.uses_barrier)
	{
		for (uint i = 0; i < count; ++i)
		{
			setInvocation(ls, gx, gy, gz, i % ls[0], (i / ls[0]) % ls[1], i / (ls[0] * ls[1]));
			s.main();
		}
		return;
	}

	static thread_local std::vector<Fiber> fibers;
	fibers.resize(count);
	ucontext_t scheduler;
	t_scheduler = &scheduler;
	t_main = s.main;
	for (uint i = 0; i < count; ++i)
	{
		Fiber& f = fibers[i];
		f.done = false;
		f.stack.resize(256 * 1024);
		getcontext(&f.ctx);
		f.ctx.uc_stack.ss_sp = f.stack.data();
		f.ctx.uc_stack.ss_size = f.stack.size();
		f.ctx.uc_link = nullptr;
		makecontext(&f.ctx, fiberEntry, 0);
	}
	// every pass resumes each live invocation once; an invocation returns here at its next barrier() or at its end
	for (bool live = true; live;)
	{
		live = false;
		for (uint i = 0; i < count; ++i)
		{
			Fiber& f = fibers[i];
			if (f.done)
				continue;
			setInvocation(ls, gx, gy, gz, i % ls[0], (i / ls[0]) % ls[1], i / (ls[0] * ls[1]));
			t_current = &f;
			swapcontext(&scheduler, &f.ctx);
			live = live || !f.done;
		}
	}
	t_scheduler = nullptr;
}

// vkCmdDispatch(x, y, z): groups spread over `threads` host threads; after(gx, gy, gz) runs on the group's thread
void dispatch(const RsShader& s, uint x, uint y, uint z, int threads, const std::function<void(uint, uint, uint)>& after = nullptr)
{
	uint64_t total = uint64_t(x) * y * z;
	if (total == 0)
		return;
	std::atomic<uint64_t> next{ 0 };
	const uint64_t chunk = 16;
	auto worker = [&]() {
		for (;;)
		{
			uint64_t b = next.fetch_add(chunk);
			if (b >= total)
				return;
			for (uint64_t g = b; g < std::min(total, b + chunk); ++g)
			{
				uint gx = uint(g % x), gy = uint((g / x) % y), gz = uint(g / (uint64_t(x) * y));
				runGroup(s, gx, gy, gz);
				if (after)
					after(gx, gy, gz);
			}
		}
	};
	int nt = int(std::min<uint64_t>(uint64_t(std::max(1, threads)), (total + chunk - 1) / chunk));
	if (nt <= 1)
		return worker();
	std::vector<std::thread> pool;
	for (int t = 0; t < nt; ++t)
		pool.emplace_back(worker);
	for (std::thread& t : pool)
		t.join();
}

glsl::texture2D pyramidView(const NvcHiZ* hiz)
{
	glsl::texture2D t = {};
	if (!hiz || !hiz->texels)
		return t;
	t.levels = hiz->levels;
	for (uint l = 0; l < hiz->levels; ++l)
	{
		t.texels[l] = hiz->texels + hiz->level_offset[l];
		t.width[l] = std::max(1u, hiz->width >> l);
		t.height[l] = std::max(1u, hiz->height >> l);
	}
	return t;
}

// Globals of meshlet.task.glsl (mesh.h): projection (unused by the task stage), CullData, screen size
struct TaskGlobals
{
	float projection[16];
	NvcCullData cullData;
	float screenWidth, screenHeight;
};

} // namespace

// the reference's mesh.h once more, only to check that the shim's types give its structs the layout of the host arrays
namespace glsl
{
namespace rs_layout
{
#include "mesh.h"
static_assert(sizeof(MeshDraw) == sizeof(NvcMeshDraw) && sizeof(Mesh) == sizeof(NvcMesh) && sizeof(MeshLod) == 20, "MeshDraw / Mesh");
static_assert(sizeof(Meshlet) == sizeof(NvcMeshlet) && sizeof(CullData) == sizeof(NvcCullData), "Meshlet / CullData");
static_assert(sizeof(MeshTaskCommand) == sizeof(NvcMeshTaskCommand) && sizeof(MeshDrawCommand) == sizeof(NvcMeshDrawCommand), "commands");
static_assert(sizeof(MeshTaskPayload) == sizeof(NvcMeshTaskPayload), "payload");
static_assert(offsetof(Globals, cullData) == 64 && offsetof(Globals, screenWidth) == 64 + sizeof(NvcCullData), "Globals");
static_assert(offsetof(Mesh, lods) == offsetof(NvcMesh, lods) && offsetof(MeshDraw, meshIndex) == offsetof(NvcMeshDraw, meshIndex), "offsets");
static_assert(offsetof(CullData, drawCount) == offsetof(NvcCullData, drawCount) && offsetof(CullData, postPass) == offsetof(NvcCullData, postPass), "CullData offsets");
} // namespace rs_layout
} // namespace glsl

namespace
{

static_assert(sizeof(glsl::float16_t) == 2, "float16_t must be storage compatible");
static_assert(sizeof(glsl::vec3) == 12 && sizeof(glsl::vec4) == 16 && sizeof(glsl::mat4) == 64, "std430 layouts used by mesh.h");

} // namespace

namespace glsl
{

void barrier()
{
	if (t_scheduler)
		swapcontext(&t_current->ctx, t_scheduler);
}

void EmitMeshTasksEXT(uint x, uint y, uint z)
{
	t_emit[0] = x;
	t_emit[1] = y;
	t_emit[2] = z;
}

void SetMeshOutputsEXT(uint vertexCount, uint primitiveCount)
{
	t_mesh_outputs[0] = vertexCount;
	t_mesh_outputs[1] = primitiveCount;
}

} // namespace glsl

extern "C"
{

// names of the shader files this library was generated from (space separated)
const char* rs_sources(void)
{
	static char buf[512];
	snprintf(buf, sizeof(buf), "%s %s %s %s %s %s %s %s", rs_shader_drawcull.source, rs_shader_tasksubmit.source, rs_shader_clustercull.source,
	    rs_shader_clustersubmit.source, rs_shader_depthreduce.source, rs_shader_meshlet_task.source, rs_shader_meshlet_mesh.source, rs_shader_mesh_vert.source);
	return buf;
}

int rs_drawcull(const NvcCullData* pass, int late, int task, const void* draws, size_t draws_bytes, const void* meshes, size_t meshes_bytes,
    uint32_t* draw_visibility, size_t dvb_bytes, void* commands, size_t commands_bytes, uint32_t* command_count4, const NvcHiZ* hiz, int threads)
{
	glsl::texture2D pyramid = pyramidView(hiz);
	if (late && pass->occlusionEnabled == 1 && pyramid.levels == 0)
		return NVC_ERROR_INVALID_ARGUMENT;

	command_count4[0] = 0; // vkCmdFillBuffer(dccb, 0, 4, 0)

	const RsShader& s = rs_shader_drawcull;
	s.spec(0, late);
	s.spec(1, task);
	s.bind(0, const_cast<void*>(draws), draws_bytes);
	s.bind(1, const_cast<void*>(meshes), meshes_bytes);
	s.bind(2, commands, commands_bytes); // DrawCommands and TaskCommands alias binding 2
	s.bind(3, command_count4, 16);
	s.bind(4, draw_visibility, dvb_bytes);
	s.bind(5, &pyramid, sizeof(pyramid));
	s.bind(6, nullptr, 0);
	s.push(pass, sizeof(*pass));
	dispatch(s, (pass->drawCount + s.local_size[0] - 1) / s.local_size[0], 1, 1, threads);

	if (task)
	{
		const RsShader& ts = rs_shader_tasksubmit;
		ts.bind(0, command_count4, 16);
		ts.bind(1, commands, commands_bytes);
		dispatch(ts, 1, 1, 1, 1);
	}
	return NVC_OK;
}

int rs_clustercull(const NvcCullData* pass, int late, const void* task_commands, size_t commands_bytes, const uint32_t* command_count4,
    const void* draws, size_t draws_bytes, const void* meshlets, size_t meshlets_bytes, uint32_t* meshlet_visibility, size_t mvb_bytes,
    uint32_t* cluster_indices, size_t cib_bytes, uint32_t* cluster_count4, const NvcHiZ* hiz, int threads)
{
	glsl::texture2D pyramid = pyramidView(hiz);
	if (late && pass->clusterOcclusionEnabled == 1 && pyramid.levels == 0)
		return NVC_ERROR_INVALID_ARGUMENT;

	cluster_count4[0] = 0; // vkCmdFillBuffer(ccb, 0, 4, 0)

	const RsShader& s = rs_shader_clustercull;
	s.spec(0, late);
	s.bind(0, const_cast<void*>(task_commands), commands_bytes);
	s.bind(1, const_cast<void*>(draws), draws_bytes);
	s.bind(2, const_cast<void*>(meshlets), meshlets_bytes);
	s.bind(3, meshlet_visibility, mvb_bytes);
	s.bind(4, &pyramid, sizeof(pyramid));
	s.bind(5, cluster_indices, cib_bytes);
	s.bind(6, cluster_count4, 16);
	s.bind(7, nullptr, 0);
	s.push(pass, sizeof(*pass));
	dispatch(s, command_count4[1], command_count4[2], command_count4[3], threads); // vkCmdDispatchIndirect(dccb, 4)

	const RsShader& cs = rs_shader_clustersubmit;
	cs.bind(0, cluster_count4, 16);
	cs.bind(1, cluster_indices, cib_bytes);
	dispatch(cs, 1, 1, 1, 1);
	return NVC_OK;
}

int rs_taskcull(const NvcCullData* pass, int late, const void* task_commands, size_t commands_bytes, const uint32_t* command_count4,
    const void* draws, size_t draws_bytes, const void* meshlets, size_t meshlets_bytes, uint32_t* meshlet_visibility, size_t mvb_bytes,
    NvcMeshTaskPayload* payloads, uint32_t* emit_counts, const NvcHiZ* hiz, int threads)
{
	glsl::texture2D pyramid = pyramidView(hiz);
	if (late && pass->clusterOcclusionEnabled == 1 && pyramid.levels == 0)
		return NVC_ERROR_INVALID_ARGUMENT;

	TaskGlobals globals = {};
	globals.cullData = *pass;

	const RsShader& s = rs_shader_meshlet_task;
	s.spec(0, late);
	s.bind(0, const_cast<void*>(task_commands), commands_bytes);
	s.bind(1, const_cast<void*>(draws), draws_bytes);
	s.bind(2, const_cast<void*>(meshlets), meshlets_bytes);
	s.bind(5, meshlet_visibility, mvb_bytes);
	s.bind(6, &pyramid, sizeof(pyramid));
	s.bind(9, nullptr, 0);
	s.push(&globals, sizeof(globals));
	uint gx = command_count4[1], gy = command_count4[2];
	dispatch(s, gx, gy, command_count4[3], threads, [&](uint x, uint y, uint) {
		uint commandId = x * 64 + y;
		emit_counts[commandId] = t_emit[0];
		memcpy(&payloads[commandId], s.payload(), sizeof(NvcMeshTaskPayload));
	});
	return NVC_OK;
}

int rs_depth_pyramid(const float* depth, uint32_t depth_width, uint32_t depth_height, const NvcHiZ* hiz, int threads)
{
	const RsShader& s = rs_shader_depthreduce;
	glsl::texture2D source = {};
	source.levels = 1;
	source.texels[0] = depth;
	source.width[0] = depth_width;
	source.height[0] = depth_height;

	for (uint32_t i = 0; i < hiz->levels; ++i)
	{
		uint32_t levelWidth = std::max(1u, hiz->width >> i), levelHeight = std::max(1u, hiz->height >> i);
		glsl::image2D target = { hiz->texels + hiz->level_offset[i], levelWidth, levelHeight };
		float reduceData[4] = { float(levelWidth), float(levelHeight), 0, 0 };

		s.bind(0, &target, sizeof(target));
		s.bind(1, &source, sizeof(source));
		s.bind(2, nullptr, 0);
		s.push(reduceData, sizeof(reduceData));
		dispatch(s, (levelWidth + s.local_size[0] - 1) / s.local_size[0], (levelHeight + s.local_size[1] - 1) / s.local_size[1], 1, threads);

		source.texels[0] = target.texels; // mipSource = mipTarget
		source.width[0] = levelWidth;
		source.height[0] = levelHeight;
	}
	return NVC_OK;
}

// ---- the consumer: meshlet.mesh.glsl (TASK = false) over the grid of vkCmdDrawMeshTasksIndirectEXT(ccb, 4) -------------
// (niagara.cpp:1655-1664: bindings dcb, db, mlb, mdb, vb, cib; push constants = Globals).  Per slot (= workgroup)
// x + 256 * y + 16 * z:   records[slot] = { vertexCount, triangleCount, out_drawId[0] (or ~0), 0 },
// positions[slot][v] = gl_MeshVerticesEXT[v].gl_Position (64 x vec4), triangles[slot][t] = gl_PrimitiveTriangleIndicesEXT[t] (96 x 3 bytes).
int rs_mesh_clusters(const float* projection16, const NvcCullData* pass, float screen_width, float screen_height, const void* task_commands,
    size_t commands_bytes, const void* draws, size_t draws_bytes, const void* meshlets, size_t meshlets_bytes, const void* meshletdata, size_t meshletdata_bytes,
    const void* vertices, size_t vertices_bytes, const uint32_t* cluster_indices, size_t cib_bytes, const uint32_t* cluster_count4, uint32_t* records, float* positions,
    uint8_t* triangles, int threads)
{
	TaskGlobals globals = {};
	memcpy(globals.projection, projection16, sizeof(globals.projection));
	globals.cullData = *pass;
	globals.screenWidth = screen_width;
	globals.screenHeight = screen_height;

	const RsShader& s = rs_shader_meshlet_mesh;
	s.spec(1, 0); // TASK = false: cluster indices come from cib
	s.bind(0, const_cast<void*>(task_commands), commands_bytes);
	s.bind(1, const_cast<void*>(draws), draws_bytes);
	s.bind(2, const_cast<void*>(meshlets), meshlets_bytes);
	s.bind(3, const_cast<void*>(meshletdata), meshletdata_bytes); // uint / uint16_t / uint8_t views alias binding 3
	s.bind(4, const_cast<void*>(vertices), vertices_bytes);
	s.bind(5, const_cast<uint32_t*>(cluster_indices), cib_bytes);
	s.push(&globals, sizeof(globals));
	dispatch(s, cluster_count4[1], cluster_count4[2], cluster_count4[3], threads, [&](uint x, uint y, uint z) {
		size_t slot = size_t(x) + size_t(y) * 256 + size_t(z) * 16; // meshlet.mesh.glsl:94
		uint vc = t_mesh_outputs[0], tc = t_mesh_outputs[1];
		const uint* drawId = static_cast<const uint*>(s.output(0));
		records[slot * 4 + 0] = vc;
		records[slot * 4 + 1] = tc;
		records[slot * 4 + 2] = vc ? drawId[0] : ~0u;
		records[slot * 4 + 3] = 0;
		for (uint v = 0; v < vc && v < 64; ++v)
			for (int c = 0; c < 4; ++c)
				positions[(slot * 64 + v) * 4 + c] = glsl::gl_MeshVerticesEXT[v].gl_Position[c];
		for (uint t = 0; t < tc && t < 96; ++t)
		{
			triangles[(slot * 96 + t) * 3 + 0] = uint8_t(glsl::gl_PrimitiveTriangleIndicesEXT[t].x);
			triangles[(slot * 96 + t) * 3 + 1] = uint8_t(glsl::gl_PrimitiveTriangleIndicesEXT[t].y);
			triangles[(slot * 96 + t) * 3 + 2] = uint8_t(glsl::gl_PrimitiveTriangleIndicesEXT[t].z);
		}
	});
	return NVC_OK;
}

// ---- the same consumer in task-shading mode (TASK = true, niagara.cpp:1666-1679): vkCmdDrawMeshTasksIndirectEXT(dccb, 4) runs
// meshlet.task per command; EmitMeshTasksEXT(n, 1, 1) then launches n mesh workgroups that read payload.clusterIndices[gl_WorkGroupID.x].
// Here the task stage's results are given (payloads[c], emit_counts[c] — from rs_taskcull, the oracle or the CUDA path) and the
// mesh stage runs over them.  Output slot s = first_slot[c] + i for the i-th mesh workgroup of command c (first_slot = exclusive
// prefix sum of emit_counts, which the caller computes); records / positions / triangles as in rs_mesh_clusters.
int rs_mesh_payloads(const float* projection16, const NvcCullData* pass, float screen_width, float screen_height, const void* task_commands,
    size_t commands_bytes, uint32_t command_count, const void* draws, size_t draws_bytes, const void* meshlets, size_t meshlets_bytes, const void* meshletdata,
    size_t meshletdata_bytes, const void* vertices, size_t vertices_bytes, const NvcMeshTaskPayload* payloads, const uint32_t* emit_counts, const uint32_t* first_slot,
    uint32_t* records, float* positions, uint8_t* triangles, int threads)
{
	TaskGlobals globals = {};
	memcpy(globals.projection, projection16, sizeof(globals.projection));
	globals.cullData = *pass;
	globals.screenWidth = screen_width;
	globals.screenHeight = screen_height;

	const RsShader& s = rs_shader_meshlet_mesh;
	s.spec(1, 1); // TASK = true: cluster indices come from the task payload
	s.bind(0, const_cast<void*>(task_commands), commands_bytes);
	s.bind(1, const_cast<void*>(draws), draws_bytes);
	s.bind(2, const_cast<void*>(meshlets), meshlets_bytes);
	s.bind(3, const_cast<void*>(meshletdata), meshletdata_bytes);
	s.bind(4, const_cast<void*>(vertices), vertices_bytes);
	s.bind(5, nullptr, 0);
	s.push(&globals, sizeof(globals));

	// one "dispatch" per task command: x = emitted mesh workgroups; the payload is the calling thread's taskPayloadSharedEXT object
	std::atomic<uint32_t> next{ 0 };
	auto worker = [&]() {
		for (uint32_t c = next.fetch_add(1); c < command_count; c = next.fetch_add(1))
		{
			uint32_t n = emit_counts[c];
			if (n > NVC_TASK_WGSIZE)
				n = NVC_TASK_WGSIZE;
			memcpy(s.payload(), &payloads[c], sizeof(NvcMeshTaskPayload));
			for (uint32_t i = 0; i < n; ++i)
			{
				runGroup(s, i, 0, 0);
				size_t slot = size_t(first_slot[c]) + i;
				uint vc = t_mesh_outputs[0], tc = t_mesh_outputs[1];
				const uint* drawId = static_cast<const uint*>(s.output(0));
				records[slot * 4 + 0] = vc;
				records[slot * 4 + 1] = tc;
				records[slot * 4 + 2] = vc ? drawId[0] : ~0u;
				records[slot * 4 + 3] = c;
				for (uint v = 0; v < vc && v < 64; ++v)
					for (int k = 0; k < 4; ++k)
						positions[(slot * 64 + v) * 4 + k] = glsl::gl_MeshVerticesEXT[v].gl_Position[k];
				for (uint t = 0; t < tc && t < 96; ++t)
				{
					triangles[(slot * 96 + t) * 3 + 0] = uint8_t(glsl::gl_PrimitiveTriangleIndicesEXT[t].x);
					triangles[(slot * 96 + t) * 3 + 1] = uint8_t(glsl::gl_PrimitiveTriangleIndicesEXT[t].y);
					triangles[(slot * 96 + t) * 3 + 2] = uint8_t(glsl::gl_PrimitiveTriangleIndicesEXT[t].z);
				}
			}
		}
	};
	int nt = std::max(1, std::min(threads, int(command_count)));
	if (nt <= 1)
		worker();
	else
	{
		std::vector<std::thread> pool;
		for (int t = 0; t < nt; ++t)
			pool.emplace_back(worker);
		for (std::thread& t : pool)
			t.join();
	}
	s.spec(1, 0);
	return NVC_OK;
}

// the test rasteriser (raster.h) over mesh-stage outputs
int rs_rasterize(const float* positions, const uint8_t* triangles, const uint32_t* records, uint32_t slots, uint32_t width, uint32_t height, float* depth,
    uint8_t* slot_hit, int mode)
{
	return rasterizeSlots(positions, triangles, records, slots, width, height, depth, slot_hit, mode);
}

// ---- the draw path's consumer: vkCmdDrawIndexedIndirectCount(dcb + 4, dccb, drawCount, 24) with mesh.vert.glsl (niagara.cpp:1680-1694) --
// For command i < command_count: indexCount indices from firstIndex, each + vertexOffset = gl_VertexIndex, gl_DrawIDARB = i; the vertex
// shader's gl_Position is rasterised as above.  mode 0: depth = max; mode 1: command_hit[i] = 1 when the command owns / ties a pixel.
int rs_draw_indexed(const float* projection16, const NvcCullData* pass, float screen_width, float screen_height, const void* draw_commands, size_t commands_bytes,
    uint32_t command_count, const void* draws, size_t draws_bytes, const void* vertices, size_t vertices_bytes, const uint32_t* indices, size_t index_count,
    uint32_t width, uint32_t height, float* depth, uint8_t* command_hit, int mode)
{
	TaskGlobals globals = {};
	memcpy(globals.projection, projection16, sizeof(globals.projection));
	globals.cullData = *pass;
	globals.screenWidth = screen_width;
	globals.screenHeight = screen_height;

	const RsShader& s = rs_shader_mesh_vert;
	s.bind(0, const_cast<void*>(draw_commands), commands_bytes);
	s.bind(1, const_cast<void*>(draws), draws_bytes);
	s.bind(2, const_cast<void*>(vertices), vertices_bytes);
	s.push(&globals, sizeof(globals));

	const NvcMeshDrawCommand* cmds = static_cast<const NvcMeshDrawCommand*>(draw_commands);
	if (size_t(command_count) * sizeof(NvcMeshDrawCommand) > commands_bytes)
		return NVC_ERROR_INVALID_ARGUMENT;
	for (uint32_t i = 0; i < command_count; ++i)
	{
		const NvcMeshDrawCommand& c = cmds[i];
		if (uint64_t(c.firstIndex) + c.indexCount > index_count)
			return NVC_ERROR_INVALID_ARGUMENT;
		for (uint32_t inst = 0; inst < c.instanceCount; ++inst)
			for (uint32_t t = 0; t + 2 < c.indexCount; t += 3)
			{
				float clip[3][4];
				const float* corner[3];
				for (int k = 0; k < 3; ++k)
				{
					glsl::gl_DrawIDARB = int(i);
					glsl::gl_VertexIndex = int(indices[c.firstIndex + t + k] + c.vertexOffset);
					s.main();
					for (int q = 0; q < 4; ++q)
						clip[k][q] = glsl::gl_Position[q];
					corner[k] = clip[k];
				}
				if (rasterTriangle(corner, width, height, depth, mode) && command_hit)
					command_hit[i] = 1;
			}
	}
	return NVC_OK;
}

// ---- math.h functions of the reference, exported for scalar cross-checks (they live in every shader TU; the
// ---- drawcull one is used) ------------------------------------------------------------------------------------------
} // extern "C"

namespace glsl
{
namespace rs_drawcull
{
bool projectSphere(vec3 c, float r, float znear, float P00, float P11, vec4& aabb);
float getOcclusionMip(vec4 aabb, float pyramidWidth, float pyramidHeight);
bool coneCull(vec3 center, float radius, vec3 cone_axis, float cone_cutoff, vec3 camera_position);
vec3 rotateQuat(vec3 v, vec4 q);
} // namespace rs_drawcull
} // namespace glsl

extern "C"
{

int rs_project_sphere(const float c[3], float r, float znear, float P00, float P11, float aabb[4])
{
	glsl::vec4 a;
	bool ok = glsl::rs_drawcull::projectSphere(glsl::vec3(c[0], c[1], c[2]), r, znear, P00, P11, a);
	if (ok)
		for (int i = 0; i < 4; ++i)
			aabb[i] = a[i];
	return ok ? 1 : 0;
}

float rs_occlusion_mip(const float aabb[4], float pw, float ph)
{
	return glsl::rs_drawcull::getOcclusionMip(glsl::vec4(aabb[0], aabb[1], aabb[2], aabb[3]), pw, ph);
}

int rs_cone_cull(const float center[3], float radius, const float axis[3], float cutoff)
{
	return glsl::rs_drawcull::coneCull(glsl::vec3(center[0], center[1], center[2]), radius, glsl::vec3(axis[0], axis[1], axis[2]), cutoff, glsl::vec3(0, 0, 0)) ? 1 : 0;
}

void rs_rotate_quat(const float v[3], const float q[4], float out[3])
{
	glsl::vec3 r = glsl::rs_drawcull::rotateQuat(glsl::vec3(v[0], v[1], v[2]), glsl::vec4(q[0], q[1], q[2], q[3]));
	out[0] = r.x;
	out[1] = r.y;
	out[2] = r.z;
}

} // extern "C"
