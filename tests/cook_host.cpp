// TEST INFRASTRUCTURE: compiles the PRODUCT's meshlet-bounds code (niagara_b200/csrc/nvc_cook.cuh, the body of
// cook_meshlet_bounds_kernel) for the host, so that the algorithm can be checked against the Meshlet[] the
// reference's cooker wrote before any GPU time is spent.  Built by tests/test_cook.py with g++ -ffp-contract=off
// into tests/_build/ (git-ignored).  Never shipped, never loaded by niagara_b200/.
#include "../niagara_b200/csrc/nvc_cook.cuh"

extern "C" int cookhost_meshlet_bounds(const NvcVertex* vertices, uint32_t vertex_count, const uint32_t* meshletdata, uint32_t meshletdata_words, NvcMeshlet* meshlets,
    uint32_t meshlet_count)
{
	(void)vertex_count;
	(void)meshletdata_words;
	for (uint32_t i = 0; i < meshlet_count; ++i)
	{
		NvcMeshlet& m = meshlets[i];
		nvc::cook::MeshletView view;
		view.vertices = vertices;
		view.data = meshletdata + m.dataOffset;
		view.baseVertex = m.baseVertex;
		view.vertexCount = m.vertexCount;
		view.triangleCount = m.triangleCount;
		view.shortRefs = m.shortRefs;
		nvc::cook::meshlet_bounds(view, &m);
	}
	return 0;
}

// the product's fp16 conversions (meshopt_quantizeHalf / meshopt_dequantizeHalf restated), for preparing test inputs
extern "C" uint16_t cookhost_quantize_half(float v)
{
	return nvc::cook::quantize_half(v);
}

extern "C" float cookhost_dequantize_half(uint16_t h)
{
	return nvc::cook::dequantize_half(h);
}
