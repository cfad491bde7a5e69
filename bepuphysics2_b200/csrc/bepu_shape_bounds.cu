// PredictBoundingBoxes kernels for every built-in shape type (sm_100a), compiled -fmad=false with IEEE div/sqrt: bit-identical to a non-contracting
// CPU evaluation of the reference's expressions (tests/test_bounds_all_shapes.py). The work is heterogeneous, so it is split by class:
//   per-body kernel  one thread per body: sleep candidacy, and the bounds of spheres, capsules, boxes, triangles and cylinders;
//   hull kernel      one warp per hull body, lane j = slot j of the reference's Vector3Wide point bundles (the reference's per-lane fold);
//   compound kernel  one warp per compound / big compound body, each lane a contiguous run of children, merged in child order;
//   mesh kernels     one CTA per chunk of up to kMeshChunkTriangles triangles (a keyed min / max reduction), then one thread per mesh body
//                    combining its chunks in order and applying the expansion.
// Every kernel reads the body's motion through load_predicted_motion, so the integrated velocity is the same bits everywhere. Bodies without a
// shape, or with a user-registered type (id > 8), get valid = 0 from the per-body kernel.
#define BEPU_NS bepu_bounds_math
#include "bepu_shape_bounds.h"
#include "bepu_bounds_motion.cuh"

namespace bepucuda {

namespace {

using namespace bepu_bounds_math;

constexpr float kMaxValue = 3.40282347e+38f;

__device__ __forceinline__ void store_bounds(float4* bounds, int body, V3 mn, V3 mx, float margin) {
    bounds[2 * (size_t)body] = make_float4(mn.x, mn.y, mn.z, margin);
    bounds[2 * (size_t)body + 1] = make_float4(mx.x, mx.y, mx.z, 1.0f);
}

__global__ void __launch_bounds__(256) shape_bounds_body_kernel(BodyBuffers B, const BodyCollidableRecord* __restrict__ collidables, BodyActivityRecord* __restrict__ activities,
                                                                float4* __restrict__ bounds, const __grid_constant__ ShapeLibraryView lib, const __grid_constant__ PredictParams p) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B.count) return;
    const PredictedMotion m = load_predicted_motion(B, i, p);
    BodyActivityRecord activity = activities[i];
    update_sleep_candidacy(activity, m.sleep_energy);
    activities[i] = activity;

    const BodyCollidableRecord c = collidables[i];
    const int32_t type = typed_index_type(c.shape);
    if (!typed_index_exists(c.shape) || type > kMesh) {
        bounds[2 * (size_t)i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        bounds[2 * (size_t)i + 1] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        return;
    }
    if (type == kConvexHull || type >= kCompound) return;  // the class kernels below
    const ConvexLocalBounds local = convex_local_bounds(lib, type, typed_index_index(c.shape), m.orientation);
    V3 mn, mx;
    float margin;
    expand_convex_bounds(local, c, m.position, m.velocity, p.dt, mn, mx, margin);
    store_bounds(bounds, i, mn, mx, margin);
}

__device__ __forceinline__ HullLane shfl_down(const HullLane& v, int offset) {
    HullLane r;
    r.min = {__shfl_down_sync(0xffffffffu, v.min.x, offset), __shfl_down_sync(0xffffffffu, v.min.y, offset), __shfl_down_sync(0xffffffffu, v.min.z, offset)};
    r.max = {__shfl_down_sync(0xffffffffu, v.max.x, offset), __shfl_down_sync(0xffffffffu, v.max.y, offset), __shfl_down_sync(0xffffffffu, v.max.z, offset)};
    r.maximumRadiusSquared = __shfl_down_sync(0xffffffffu, v.maximumRadiusSquared, offset);
    return r;
}
__device__ __forceinline__ MergedBounds shfl_down(const MergedBounds& v, int offset) {
    MergedBounds r;
    r.min = {__shfl_down_sync(0xffffffffu, v.min.x, offset), __shfl_down_sync(0xffffffffu, v.min.y, offset), __shfl_down_sync(0xffffffffu, v.min.z, offset)};
    r.max = {__shfl_down_sync(0xffffffffu, v.max.x, offset), __shfl_down_sync(0xffffffffu, v.max.y, offset), __shfl_down_sync(0xffffffffu, v.max.z, offset)};
    r.speculativeMargin = __shfl_down_sync(0xffffffffu, v.speculativeMargin, offset);
    return r;
}

// Offsets 1, 2, 4, ...: every step merges two ADJACENT runs of lanes, the lower run as `running`, so lane 0 ends with the fold in lane order.
__global__ void __launch_bounds__(256) shape_bounds_hull_kernel(BodyBuffers B, const BodyCollidableRecord* __restrict__ collidables, const int32_t* __restrict__ bodies, int32_t count,
                                                                float4* __restrict__ bounds, const __grid_constant__ ShapeLibraryView lib, const __grid_constant__ PredictParams p) {
    const int w = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = (int)(threadIdx.x & 31);
    if (w >= count) return;  // whole warps leave together
    const int body = bodies[w];
    const PredictedMotion m = load_predicted_motion(B, body, p);
    const BodyCollidableRecord c = collidables[body];
    const HullRecord hull = lib.hulls[typed_index_index(c.shape)];
    HullLane folded = {{kMaxValue, kMaxValue, kMaxValue}, {-kMaxValue, -kMaxValue, -kMaxValue}, 0.0f};
    if (lane < lib.hull_width) folded = hull_lane_fold(lib.hull_points, lib.hull_width, hull, lane, matrix_from_quaternion(m.orientation));
    for (int offset = 1; offset < 32; offset <<= 1) {
        const HullLane higher = shfl_down(folded, offset);
        if ((lane & (2 * offset - 1)) == 0) hull_lane_merge(folded, higher);
    }
    if (lane == 0) {
        V3 mn, mx;
        float margin;
        expand_convex_bounds(hull_finish(folded), c, m.position, m.velocity, p.dt, mn, mx, margin);
        store_bounds(bounds, body, mn, mx, margin);
    }
}

__global__ void __launch_bounds__(256) shape_bounds_compound_kernel(BodyBuffers B, const BodyCollidableRecord* __restrict__ collidables, const int32_t* __restrict__ bodies, int32_t count,
                                                                    float4* __restrict__ bounds, const __grid_constant__ ShapeLibraryView lib, const __grid_constant__ PredictParams p) {
    const int w = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = (int)(threadIdx.x & 31);
    if (w >= count) return;
    const int body = bodies[w];
    const PredictedMotion m = load_predicted_motion(B, body, p);
    const BodyCollidableRecord c = collidables[body];
    const CompoundRecord compound = (typed_index_type(c.shape) == kCompound ? lib.compounds : lib.big_compounds)[typed_index_index(c.shape)];
    // lane l takes children [l * per, (l + 1) * per): contiguous runs, so merging lanes in order is merging children in order
    const int per = (compound.child_count + 31) >> 5;
    const int begin = min(lane * per, compound.child_count), end = min(begin + per, compound.child_count);
    MergedBounds merged = merged_bounds_start();
    for (int k = begin; k < end; ++k)
        merge_bounds(merged, compound_child_bounds(lib, lib.compound_children[(size_t)compound.first_child + k], c, m.orientation, m.position, m.velocity, p.dt));
    for (int offset = 1; offset < 32; offset <<= 1) {
        const MergedBounds later = shfl_down(merged, offset);
        if ((lane & (2 * offset - 1)) == 0) merge_bounds(merged, later);
    }
    if (lane == 0) store_bounds(bounds, body, merged.min, merged.max, merged.speculativeMargin);
}

struct Keyed6 {
    float v[6];  // min.xyz, max.xyz
    int32_t k[6];
};
__device__ __forceinline__ void combine(Keyed6& a, const Keyed6& b) {
    for (int d = 0; d < 3; ++d) mesh_combine_min(a.v[d], a.k[d], b.v[d], b.k[d]);
    for (int d = 3; d < 6; ++d) mesh_combine_max(a.v[d], a.k[d], b.v[d], b.k[d]);
}

// One CTA per chunk: each thread folds the triangles t, t + 256, ... of the chunk in order (the reference's step, keyed by triangle), then the
// CTA combines the (value, triangle) pairs; the smaller triangle index wins a tie, which is what the sequential fold keeps.
__global__ void __launch_bounds__(256) shape_bounds_mesh_chunk_kernel(BodyBuffers B, const MeshBody* __restrict__ meshBodies, const MeshChunk* __restrict__ chunks,
                                                                      float* __restrict__ partials, const __grid_constant__ ShapeLibraryView lib) {
    __shared__ Keyed6 warpResults[8];
    const MeshChunk chunk = chunks[blockIdx.x];
    const MeshBody mb = meshBodies[chunk.mesh_body];
    const MeshRecord mesh = lib.meshes[mb.mesh];
    const float4 q4 = B.pose[2 * (size_t)mb.body];
    const M33 r = narrow_matrix_from_quaternion(Q4{q4.x, q4.y, q4.z, q4.w});
    const V3 scale = {mesh.scale[0], mesh.scale[1], mesh.scale[2]};
    Keyed6 acc;
    for (int d = 0; d < 6; ++d) acc.v[d] = d < 3 ? kMaxValue : -kMaxValue, acc.k[d] = INT32_MAX;
    const float* triangles = lib.mesh_triangles + 9 * (size_t)chunk.first_triangle;
    for (int t = threadIdx.x; t < chunk.triangle_count; t += blockDim.x) {
        V3 a, b, c;
        mesh_triangle_vertices(triangles + 9 * (size_t)t, scale, r, a, b, c);
        mesh_fold_min(a.x, b.x, c.x, t, acc.v[0], acc.k[0]);
        mesh_fold_min(a.y, b.y, c.y, t, acc.v[1], acc.k[1]);
        mesh_fold_min(a.z, b.z, c.z, t, acc.v[2], acc.k[2]);
        mesh_fold_max(a.x, b.x, c.x, t, acc.v[3], acc.k[3]);
        mesh_fold_max(a.y, b.y, c.y, t, acc.v[4], acc.k[4]);
        mesh_fold_max(a.z, b.z, c.z, t, acc.v[5], acc.k[5]);
    }
    for (int offset = 16; offset > 0; offset >>= 1) {
        Keyed6 other;
        for (int d = 0; d < 6; ++d) other.v[d] = __shfl_down_sync(0xffffffffu, acc.v[d], offset), other.k[d] = __shfl_down_sync(0xffffffffu, acc.k[d], offset);
        combine(acc, other);
    }
    if ((threadIdx.x & 31) == 0) warpResults[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int wi = 1; wi < (int)(blockDim.x >> 5); ++wi) combine(acc, warpResults[wi]);
        for (int d = 0; d < 6; ++d) partials[6 * (size_t)blockIdx.x + d] = acc.v[d];
    }
}

// One thread per mesh body: the chunks in order (a tie keeps the earlier chunk, as the sequential fold keeps the earlier triangle), then
// ExecuteHomogeneousCompoundBatch's expansion.
__global__ void __launch_bounds__(128) shape_bounds_mesh_finish_kernel(BodyBuffers B, const BodyCollidableRecord* __restrict__ collidables, const MeshBody* __restrict__ meshBodies,
                                                                       int32_t count, const float* __restrict__ partials, float4* __restrict__ bounds, const __grid_constant__ PredictParams p) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const MeshBody mb = meshBodies[i];
    const PredictedMotion m = load_predicted_motion(B, mb.body, p);
    V3 mn = {kMaxValue, kMaxValue, kMaxValue}, mx = {-kMaxValue, -kMaxValue, -kMaxValue};
    for (int k = 0; k < mb.chunk_count; ++k) {
        const float* part = partials + 6 * ((size_t)mb.first_chunk + k);
        mn = vmin3(V3{part[0], part[1], part[2]}, mn);
        mx = vmax3(V3{part[3], part[4], part[5]}, mx);
    }
    V3 boundsMin, boundsMax;
    float margin;
    mesh_bounds(mn, mx, collidables[mb.body], m.position, m.velocity, p.dt, boundsMin, boundsMax, margin);
    store_bounds(bounds, mb.body, boundsMin, boundsMax, margin);
}

}  // namespace

void launch_predict_shape_bounds(const BodyBuffers& B, const ShapeLibraryView& library, const ShapeBoundsWork& work, BodyActivityRecord* activities, float4* bounds,
                                 const PredictParams& params, cudaStream_t s) {
    if (B.count <= 0) return;
    shape_bounds_body_kernel<<<(unsigned)((B.count + 255) / 256), 256, 0, s>>>(B, work.collidables, activities, bounds, library, params);
    if (work.hull_body_count > 0)
        shape_bounds_hull_kernel<<<(unsigned)((work.hull_body_count + 7) / 8), 256, 0, s>>>(B, work.collidables, work.hull_bodies, work.hull_body_count, bounds, library, params);
    if (work.compound_body_count > 0)
        shape_bounds_compound_kernel<<<(unsigned)((work.compound_body_count + 7) / 8), 256, 0, s>>>(B, work.collidables, work.compound_bodies, work.compound_body_count, bounds, library,
                                                                                                   params);
    if (work.mesh_chunk_count > 0) {
        shape_bounds_mesh_chunk_kernel<<<(unsigned)work.mesh_chunk_count, 256, 0, s>>>(B, work.mesh_bodies, work.mesh_chunks, work.mesh_partials, library);
        shape_bounds_mesh_finish_kernel<<<(unsigned)((work.mesh_body_count + 127) / 128), 128, 0, s>>>(B, work.collidables, work.mesh_bodies, work.mesh_body_count, work.mesh_partials,
                                                                                                      bounds, params);
    }
}

}  // namespace bepucuda
