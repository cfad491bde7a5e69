// PredictBoundingBoxes on the device for every built-in shape type (bepucuda_set_shape_library / bepucuda_set_body_collidables): the per-class
// launches of bepu_shape_bounds.cu and the work lists the host builds for them.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

#include "bepu_bounds.h"
#include "bepu_device_types.h"
#ifndef BEPU_NS
#define BEPU_NS bepu_bounds_math  // the namespace bepu_bounds.cu and bepu_shape_bounds.cu compile the bounds arithmetic into
#endif
#include "bepu_shape_bounds_math.cuh"

namespace bepucuda {

using bepu_bounds_math::BodyCollidableRecord;
using bepu_bounds_math::ShapeLibraryView;

// Triangles per CTA of the mesh pass: a mesh with more is spread over several CTAs, whose partial boxes a second pass combines in chunk order.
constexpr int kMeshChunkTriangles = 8192;

struct MeshChunk {
    int64_t first_triangle;  // into the mesh triangle pool
    int32_t triangle_count;
    int32_t mesh_body;       // index into ShapeBoundsWork::mesh_bodies
};
struct MeshBody {
    int32_t body, mesh, first_chunk, chunk_count;
};

struct ShapeBoundsWork {
    const BodyCollidableRecord* collidables;  // one per body
    const int32_t* hull_bodies;               // bodies whose shape is a convex hull (type 5)
    const int32_t* compound_bodies;           // compounds and big compounds (types 6, 7)
    const MeshBody* mesh_bodies;              // meshes (type 8)
    const MeshChunk* mesh_chunks;
    float* mesh_partials;                     // 6 floats per chunk: min.xyz, max.xyz
    int32_t hull_body_count, compound_body_count, mesh_body_count, mesh_chunk_count;
};

// Issues, on stream s, the per-body kernel (activity, primitives, triangles) and then the hull, compound and mesh kernels that have work.
// bounds: 8 floats per body {min.xyz, speculative margin, max.xyz, valid}.
void launch_predict_shape_bounds(const BodyBuffers& B, const ShapeLibraryView& library, const ShapeBoundsWork& work, BodyActivityRecord* activities, float4* bounds,
                                 const PredictParams& params, cudaStream_t s);

}  // namespace bepucuda
